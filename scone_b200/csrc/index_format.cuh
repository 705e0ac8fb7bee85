// index_format.cuh -- the device side of the f-gram index's slot formats (index_plan.h): the index handle and the view the
// kernels read, the pre-filter, and the one probe and one insert of every format.  A key is the f-gram's tokens in REVERSE
// reading order (key[0] = last token), -1 padded to seven; its home slot comes from the rolling hash of common.cuh.
#pragma once
#include "common.cuh"
#include "index_plan.h"

namespace scone {

// device view passed by value to kernels
struct IndexView {
    void *slots;  // `cap` slots of `format`
    uint64_t cap;
    uint32_t len_mask;
    int32_t max_n;
    SlotFormat format;
    uint32_t *filter;      // pre-filter words (see filter_pass), or NULL = probe every candidate
    uint32_t filter_mask;  // number of words (any count: the word is picked by a multiply-high, not a mask)
};

struct scone_index_impl {
    IndexView v;  // with the filter, whatever the batch size (view_of)
    int64_t n;
    int32_t max_probe;
    int32_t filter_always;  // SCONE_INDEX_FILTER=always: consult the filter for every batch size (testing)
};

// Batches below this many positions are latency-bound: the filter's extra L2 round trip costs more than the probes it saves.
constexpr int64_t kFilterMinPositions = 16384;

// the view a batch of `positions` positions reads
inline IndexView view_of(const scone_index_impl *ix, int64_t positions) {
    IndexView v = ix->v;
    if (!ix->filter_always && positions < kFilterMinPositions) v.filter = nullptr;
    return v;
}

// Pre-filter (sized by plan_index): a blocked Bloom filter, two bits (hash bits 32-41) of one word (multiply-high of the low
// 32 bits) per key.  Most candidate n-grams are NOT in the vocabulary: answering those from L2 instead of with a random
// 64-byte DRAM read of a slot takes two thirds of the probe traffic away from the row gather.
__host__ __device__ __forceinline__ uint32_t filter_bits(uint64_t h) {
    return (1u << (uint32_t)((h >> 32) & 31u)) | (1u << (uint32_t)((h >> 37) & 31u));
}

__host__ __device__ __forceinline__ uint32_t filter_word(uint64_t h, uint32_t words) {
    return (uint32_t)(((uint64_t)(uint32_t)h * (uint64_t)words) >> 32);
}

__device__ __forceinline__ bool filter_pass(const IndexView &ix, uint64_t h) {
    if (!ix.filter) return true;
    uint32_t w;
    // (L2 default priority is enough: everything streamed is evict-first; the .L2::evict_last form exists for 256-bit loads only)
    asm volatile("ld.global.nc.L1::evict_last.b32 %0, [%1];" : "=r"(w) : "l"(ix.filter + filter_word(h, ix.filter_mask)));
    const uint32_t b = filter_bits(h);
    return (w & b) == b;
}

// The formats: `pack` puts a key into its slot's words (k[0]: the key's bits of the first word, ORed into the id) and says
// whether it fits, `empty` tests a first word, `match` compares a slot with a packed key, `id` reads a matching slot's id.
// Empty slots are all-ones bytes in every format, yet the empty tests differ: one shared test changes the probe's code.
template <SlotFormat FMT>
struct SlotOf {
    static constexpr SlotFormat kFormat = FMT;
    static constexpr int kWords = kSlotFormats[FMT].slot_bytes / 4, kPerStep = kProbeStepBytes / kSlotFormats[FMT].slot_bytes;
    static __device__ __forceinline__ bool empty(int32_t w0) { return w0 < 0; }
    static __device__ __forceinline__ int32_t id(int32_t w0) { return w0; }
};

// w[0] = id, w[1..7] = the key.  Tokens are non-negative, so the -1 padding encodes the length and equality of the seven
// words is exact equality of (length, tokens): no verify read, no 64-bit-hash aliasing.
struct WideSlot : SlotOf<kSlotWide> {
    static_assert(kWords == 8 && kSlotFormats[kFormat].max_n == 7, "id + seven int32 tokens");
    static __device__ __forceinline__ bool pack(const int32_t (&key)[7], uint32_t (&k)[kWords]) {
        k[0] = 0;
#pragma unroll
        for (int i = 0; i < 7; ++i) k[i + 1] = (uint32_t)key[i];
        return true;
    }
    static __device__ __forceinline__ bool match(const int32_t *w, const uint32_t (&k)[kWords]) {
        bool eq = true;
#pragma unroll
        for (int i = 1; i < kWords; ++i) eq &= (w[i] == (int32_t)k[i]);
        return eq;
    }
};

// w[0] = id, w[1 + i] = key[2i] | key[2i + 1] << 16, 0xFFFF padded.
struct Compact16Slot : SlotOf<kSlotCompact16> {
    static constexpr int32_t kPad = 0xFFFF;
    static_assert(kWords == 4 && kSlotFormats[kFormat].max_n == 6 && kPad == kSlotFormats[kFormat].tok_limit, "id + six 16-bit tokens");
    static __device__ __forceinline__ bool pack(const int32_t (&key)[7], uint32_t (&k)[kWords]) {
        k[0] = 0;
        bool ok = key[6] < 0;
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            const int32_t lo = key[2 * i], hi = key[2 * i + 1];
            ok = ok && lo < kPad && hi < kPad;
            k[i + 1] = (uint32_t)(lo < 0 ? kPad : lo) | ((uint32_t)(hi < 0 ? kPad : hi) << 16);
        }
        return ok;
    }
    static __device__ __forceinline__ bool match(const int32_t *w, const uint32_t (&k)[kWords]) {
        return (uint32_t)w[1] == k[1] && (uint32_t)w[2] == k[2] && (uint32_t)w[3] == k[3];
    }
};

// tokens t0..t4 0xFFFFF padded; w0 is all-ones only for an id no vocabulary has (n_limit):
//   w0 = id | t0[3:0] << 28      w1 = t0[19:4] | t1[15:0] << 16      w2 = t1[19:16] | t2 << 4 | t3[7:0] << 24      w3 = t3[19:8] | t4 << 12
struct Compact20Slot : SlotOf<kSlotCompact20> {
    static constexpr uint32_t kPad = 0xFFFFFu, kIdMask = 0x0FFFFFFFu;
    static_assert(kWords == 4 && kSlotFormats[kFormat].max_n == 5 && kPad == kSlotFormats[kFormat].tok_limit &&
                  kIdMask == kSlotFormats[kFormat].n_limit, "28-bit id + five 20-bit tokens");
    static __device__ __forceinline__ bool pack(const int32_t (&key)[7], uint32_t (&k)[kWords]) {
        bool ok = key[5] < 0 && key[6] < 0;
        uint32_t t[5];
#pragma unroll
        for (int i = 0; i < 5; ++i) {
            ok = ok && key[i] < (int32_t)kPad;
            t[i] = key[i] < 0 ? kPad : (uint32_t)key[i];
        }
        k[0] = (t[0] & 0xFu) << 28;
        k[1] = (t[0] >> 4) | ((t[1] & 0xFFFFu) << 16);
        k[2] = (t[1] >> 16) | (t[2] << 4) | ((t[3] & 0xFFu) << 24);
        k[3] = (t[3] >> 8) | (t[4] << 12);
        return ok;
    }
    static __device__ __forceinline__ bool empty(int32_t w0) { return (uint32_t)w0 == ~0u; }
    static __device__ __forceinline__ bool match(const int32_t *w, const uint32_t (&k)[kWords]) {
        return ((uint32_t)w[0] & ~kIdMask) == k[0] && (uint32_t)w[1] == k[1] && (uint32_t)w[2] == k[2] && (uint32_t)w[3] == k[3];
    }
    static __device__ __forceinline__ int32_t id(int32_t w0) { return (int32_t)((uint32_t)w0 & kIdMask); }
};

template <class F>
__device__ __forceinline__ uint64_t home_slot(uint64_t h, uint64_t cap) { return __umul64hi(h, cap / F::kPerStep) * F::kPerStep; }

// 256-bit load of half a probe step (.nc: no build runs during a lookup), evict-last: every batch re-reads the index
__device__ __forceinline__ void load_slot(const int32_t *p, int32_t (&w)[8]) {
    asm volatile("ld.global.nc.L1::evict_last.L2::evict_last.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(w[0]), "=r"(w[1]), "=r"(w[2]), "=r"(w[3]), "=r"(w[4]), "=r"(w[5]), "=r"(w[6]), "=r"(w[7])
                 : "l"(p));
}

// The f-gram id of `key`, or -1.  The insert fills s, s+1, s+2, ... from the home slot on, so walking the slots of each block
// in order is exact: the first empty slot ends the chain.
template <class F>
__device__ __forceinline__ int32_t probe(const IndexView &ix, uint64_t h, const int32_t (&key)[7]) {
    uint32_t k[F::kWords];
    if (!F::pack(key, k)) return -1;  // a key the format cannot hold is not in the vocabulary
    const int32_t *slots = static_cast<const int32_t *>(ix.slots);
    uint64_t s = home_slot<F>(h, ix.cap);
    for (uint64_t it = 0; it < ix.cap; it += F::kPerStep) {
        int32_t a[8], b[8];  // slots s .. s + kPerStep - 1
        load_slot(slots + s * F::kWords, a);
        load_slot(slots + s * F::kWords + 8, b);
        if constexpr (F::kPerStep == 2) {
            // written out: as a two-trip loop the walk compiles to a probe that loads b only after a's compare, and spills
            if (F::empty(a[0])) return -1;
            if (F::match(a, k)) return F::id(a[0]);
            if (F::empty(b[0])) return -1;
            if (F::match(b, k)) return F::id(b[0]);
        } else {
#pragma unroll
            for (int q = 0; q < F::kPerStep; ++q) {
                const int32_t *w = (q * F::kWords < 8 ? a : b) + q * F::kWords % 8;
                if (F::empty(w[0])) return -1;
                if (F::match(w, k)) return F::id(w[0]);
            }
        }
        s += F::kPerStep;
        if (s == ix.cap) s = 0;
    }
    return -1;
}

// Claims the first free slot from the home slot on (CAS of its first word) and writes the rest of the key; returns the slots
// tried.  The key fits (the scan and plan_index saw to that), and no lookup runs concurrently.
template <class F>
__device__ __forceinline__ int insert(void *slots, uint64_t cap, uint64_t h, const int32_t (&key)[7], uint32_t id) {
    uint32_t k[F::kWords];
    F::pack(key, k);
    uint32_t *words = static_cast<uint32_t *>(slots);
    uint64_t s = home_slot<F>(h, cap);
    int probes = 1;
    for (; atomicCAS(words + s * F::kWords, ~0u, id | k[0]) != ~0u; ++probes)
        if (++s == cap) s = 0;
#pragma unroll
    for (int j = 1; j < F::kWords; ++j) words[s * F::kWords + j] = k[j];
    return probes;
}

__device__ __forceinline__ int32_t probe_any(const IndexView &ix, uint64_t h, const int32_t (&key)[7]) {
    if (!filter_pass(ix, h)) return -1;
    return ix.format == kSlotCompact16   ? probe<Compact16Slot>(ix, h, key)
           : ix.format == kSlotCompact20 ? probe<Compact20Slot>(ix, h, key)
                                         : probe<WideSlot>(ix, h, key);
}

}  // namespace scone
