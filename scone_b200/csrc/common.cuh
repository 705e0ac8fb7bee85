// common.cuh -- shared device/host helpers for libscone_b200 (sm_100a only).
#pragma once

#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <cstdarg>
#include <cstdio>

#include "../../include/scone_b200.h"

// ---------------------------------------------------------------------------------------------
// host side: error plumbing (no exceptions cross the C ABI)
// ---------------------------------------------------------------------------------------------
namespace scone {

void set_error(const char *fmt, ...);
extern std::atomic<int64_t> g_launches;

#define SCONE_CUDA(expr)                                                                              \
    do {                                                                                              \
        cudaError_t _e = (expr);                                                                      \
        if (_e != cudaSuccess) {                                                                      \
            ::scone::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
            return SCONE_E_CUDA;                                                                      \
        }                                                                                             \
    } while (0)

#define SCONE_REQUIRE(cond, ...)              \
    do {                                      \
        if (!(cond)) {                        \
            ::scone::set_error(__VA_ARGS__);  \
            return SCONE_E_INVALID;           \
        }                                     \
    } while (0)

// after a <<<>>> launch
#define SCONE_LAUNCHED()                 \
    do {                                 \
        ::scone::g_launches.fetch_add(1); \
        SCONE_CUDA(cudaGetLastError());  \
    } while (0)

constexpr int kNumSMsB200 = 148;

// 1-D grid size for `count` blocks; a count beyond the hardware limit is an error, not a silently truncated grid
#define SCONE_GRID(var, count, who)                                                                              \
    const int64_t var##_i64 = (count);                                                                           \
    SCONE_REQUIRE(var##_i64 <= 0x7FFFFFFFll, "%s: %lld thread blocks exceed the grid limit (split the call)", who, \
                  (long long)var##_i64);                                                                         \
    const unsigned var = (unsigned)var##_i64

// ---------------------------------------------------------------------------------------------
// index slot format: 32 bytes = one DRAM sector.
//   w[0]    f-gram id, -1 = empty
//   w[1..7] tokens in REVERSE reading order (w[1] = last token), -1 padded.  Token ids are
//           non-negative int32, so the padding also encodes the length and equality of the seven
//           words is exact equality of (length, tokens): no verify read, no 64-bit-hash aliasing.
// ---------------------------------------------------------------------------------------------
struct __align__(32) Slot {
    int32_t w[8];
};
static_assert(sizeof(Slot) == 32, "slot must be one sector");

// Compact slot format, used when every vocabulary token is < 65535 and max_n <= 6 (e.g. GPT-2's 50 257 tokens):
// 16 bytes = id + six 16-bit tokens (reverse order, 0xFFFF padded).  Four slots per 64-byte block, half the index
// bytes per f-gram: a 1 M f-gram index is 32 MB at load factor 0.5 and stays resident in the 126 MB L2.
struct __align__(16) Slot16 {
    int32_t id;
    uint32_t t[3];
};
static_assert(sizeof(Slot16) == 16, "compact slot");

// Second compact format, for vocabularies whose tokens do not fit 16 bits (V = 128 000: configs 3-5): 16 bytes = a 28-bit
// id + FIVE 20-bit tokens (reverse order, 0xFFFFF padded); needs max_n <= 5, tokens < 1 048 575 and fewer than 2^28 - 1
// f-grams.  Same 64-byte probe step of four slots; the all-ones first word marks an empty slot.
//   w0 = id | t0[3:0] << 28      w1 = t0[19:4] | t1[15:0] << 16      w2 = t1[19:16] | t2 << 4 | t3[7:0] << 24      w3 = t3[19:8] | t4 << 12
struct __align__(16) Slot20 {
    uint32_t w[4];
};
static_assert(sizeof(Slot20) == 16, "compact-20 slot");
constexpr uint32_t kPad20 = 0xFFFFFu, kEmpty20 = 0xFFFFFFFFu, kIdMask20 = 0x0FFFFFFFu;

enum SlotFormat : int32_t { kSlotWide = 0, kSlotCompact16 = 1, kSlotCompact20 = 2 };

struct scone_index_impl {
    Slot *slots;  // Slot, Slot16 or Slot20 array, `cap` entries
    uint64_t cap;
    int64_t n;
    int32_t max_n;
    uint32_t len_mask;
    int32_t max_probe;
    int32_t compact;  // SlotFormat
    int device;
    uint32_t *filter;      // pre-filter words (see filter_pass), or NULL
    uint32_t filter_mask;  // number of words (any count: the word is picked by a multiply-high, not a mask)
    int32_t filter_always; // SCONE_INDEX_FILTER=always: consult it for every batch size (testing)
};

// device view passed by value to kernels
struct IndexView {
    const Slot *slots;
    uint64_t cap;
    uint32_t len_mask;
    int32_t max_n;
    int32_t compact;
    const uint32_t *filter;  // NULL = probe every candidate
    uint32_t filter_mask;    // number of filter words
};

// Batches below this many positions are latency-bound: the filter's extra L2 round trip costs more than the probes it saves.
constexpr int64_t kFilterMinPositions = 16384;

inline IndexView view_of(const scone_index_impl *ix, int64_t positions) {
    const bool use = ix->filter && (ix->filter_always || positions >= kFilterMinPositions);
    return IndexView{ix->slots, ix->cap, ix->len_mask, ix->max_n, ix->compact, use ? ix->filter : nullptr, ix->filter_mask};
}

// ---------------------------------------------------------------------------------------------
// rolling 64-bit hash of the n-gram ENDING at a position: tokens are folded last-to-first, so
// the hash of the (n+1)-gram is one step on from the hash of the n-gram with the same end.
// ---------------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ uint64_t hash_seed() { return 0x243F6A8885A308D3ull; }

__host__ __device__ __forceinline__ uint64_t hash_roll(uint64_t h, uint32_t tok) {
    h = (h ^ (uint64_t)tok) * 0x9E3779B97F4A7C15ull;
    return h ^ (h >> 29);
}

__host__ __device__ __forceinline__ uint64_t hash_finish(uint64_t h, int n) {
    h ^= (uint64_t)n * 0xD6E8FEB86659FD93ull;
    h ^= h >> 33;
    h *= 0xFF51AFD7ED558CCDull;
    h ^= h >> 33;
    h *= 0xC4CEB9FE1A85EC53ull;
    h ^= h >> 33;
    return h;
}

#ifdef __CUDACC__

// Home slots are EVEN: a probe step reads the aligned pair (s, s+1) = one 64-byte block, which is what a DRAM access
// fetches anyway, so checking two slots per dependent step is free in traffic and halves the probe chain.
// (capacity is a multiple of 4.)
__device__ __forceinline__ uint64_t home_slot(uint64_t h, uint64_t cap) { return __umul64hi(h, cap >> 1) << 1; }

// 256-bit slot load (LDG.E.256); slots are read-only while any lookup runs.
__device__ __forceinline__ void load_slot(const Slot *p, int32_t (&w)[8]) {
    // evict-last in L1 and L2: the index is re-read by every batch, the streamed rows are not
    asm volatile("ld.global.nc.L1::evict_last.L2::evict_last.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(w[0]), "=r"(w[1]), "=r"(w[2]), "=r"(w[3]), "=r"(w[4]), "=r"(w[5]), "=r"(w[6]), "=r"(w[7])
                 : "l"(p));
}

// key[0..6]: reversed tokens, -1 padded.  Returns the f-gram id or -1.
__device__ __forceinline__ int32_t probe(const IndexView &ix, uint64_t h, const int32_t (&key)[7]) {
    uint64_t s = home_slot(h, ix.cap);  // even; the insert order is s, s+1, s+2, ... so scanning pairs in order is exact
    for (uint64_t it = 0; it < ix.cap; it += 2) {
        int32_t a[8], b[8];
        load_slot(ix.slots + s, a);
        load_slot(ix.slots + s + 1, b);
        if (a[0] < 0) return -1;
        bool eq = true;
#pragma unroll
        for (int k = 0; k < 7; ++k) eq &= (a[k + 1] == key[k]);
        if (eq) return a[0];
        if (b[0] < 0) return -1;
        eq = true;
#pragma unroll
        for (int k = 0; k < 7; ++k) eq &= (b[k + 1] == key[k]);
        if (eq) return b[0];
        s += 2;
        if (s == ix.cap) s = 0;
    }
    return -1;
}

// compact format: home slots are multiples of 4, a probe step reads the whole 64-byte block (four slots)
__device__ __forceinline__ uint64_t home_slot16(uint64_t h, uint64_t cap) { return __umul64hi(h, cap >> 2) << 2; }

__device__ __forceinline__ bool pack_key16(const int32_t (&key)[7], uint32_t (&k)[3]) {
    bool ok = key[6] < 0;  // at most six tokens
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        const int32_t lo = key[2 * i], hi = key[2 * i + 1];
        ok = ok && lo < 0xFFFF && hi < 0xFFFF;
        k[i] = (uint32_t)(lo < 0 ? 0xFFFF : lo) | ((uint32_t)(hi < 0 ? 0xFFFF : hi) << 16);
    }
    return ok;
}

__device__ __forceinline__ int32_t probe16(const IndexView &ix, uint64_t h, const int32_t (&key)[7]) {
    uint32_t k[3];
    if (!pack_key16(key, k)) return -1;  // a token >= 65535 cannot be in a compact vocabulary
    const Slot16 *slots = reinterpret_cast<const Slot16 *>(ix.slots);
    uint64_t s = home_slot16(h, ix.cap);
    for (uint64_t it = 0; it < ix.cap; it += 4) {
        int32_t a[8], b[8];
        load_slot(reinterpret_cast<const Slot *>(slots + s), a);      // slots s, s+1
        load_slot(reinterpret_cast<const Slot *>(slots + s + 2), b);  // slots s+2, s+3
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int32_t *w = (q < 2 ? a : b) + 4 * (q & 1);
            if (w[0] < 0) return -1;
            if ((uint32_t)w[1] == k[0] && (uint32_t)w[2] == k[1] && (uint32_t)w[3] == k[2]) return w[0];
        }
        s += 4;
        if (s == ix.cap) s = 0;
    }
    return -1;
}

__device__ __forceinline__ bool pack_key20(const int32_t (&key)[7], uint32_t (&k)[4]) {
    bool ok = key[5] < 0 && key[6] < 0;  // at most five tokens
    uint32_t t[5];
#pragma unroll
    for (int i = 0; i < 5; ++i) {
        ok = ok && key[i] < (int32_t)kPad20;
        t[i] = key[i] < 0 ? kPad20 : (uint32_t)key[i];
    }
    k[0] = (t[0] & 0xFu) << 28;  // compared with the top four bits of w0
    k[1] = (t[0] >> 4) | ((t[1] & 0xFFFFu) << 16);
    k[2] = (t[1] >> 16) | (t[2] << 4) | ((t[3] & 0xFFu) << 24);
    k[3] = (t[3] >> 8) | (t[4] << 12);
    return ok;
}

__device__ __forceinline__ int32_t probe20(const IndexView &ix, uint64_t h, const int32_t (&key)[7]) {
    uint32_t k[4];
    if (!pack_key20(key, k)) return -1;  // a token >= 2^20 - 1 or a sixth token cannot be in a compact-20 vocabulary
    const Slot20 *slots = reinterpret_cast<const Slot20 *>(ix.slots);
    uint64_t s = home_slot16(h, ix.cap);
    for (uint64_t it = 0; it < ix.cap; it += 4) {
        int32_t a[8], b[8];
        load_slot(reinterpret_cast<const Slot *>(slots + s), a);      // slots s, s+1
        load_slot(reinterpret_cast<const Slot *>(slots + s + 2), b);  // slots s+2, s+3
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int32_t *w = (q < 2 ? a : b) + 4 * (q & 1);
            if ((uint32_t)w[0] == kEmpty20) return -1;
            if (((uint32_t)w[0] & ~kIdMask20) == k[0] && (uint32_t)w[1] == k[1] && (uint32_t)w[2] == k[2] && (uint32_t)w[3] == k[3])
                return (int32_t)((uint32_t)w[0] & kIdMask20);
        }
        s += 4;
        if (s == ix.cap) s = 0;
    }
    return -1;
}

// ---------------------------------------------------------------------------------------------
// Pre-filter: 16 bits of a blocked Bloom filter per f-gram (two bits of one 32-bit word per key, ~1.5 % false
// positives, no false negatives).  For vocabularies of a few million f-grams it stays resident in L2, and most candidate
// n-grams of a position are NOT in the vocabulary: answering those from L2 instead of with a random 64-byte DRAM read of
// a slot takes two thirds of the probe traffic (and DRAM row activations) away from the row gather they compete with.
// The word index is a multiply-high of the low 32 hash bits with the word count (any count, so the filter is exactly as
// large as its bits-per-key budget asks), the bit positions come from bits 32-41; the home slot from the top bits.
// Vocabularies of up to 12 M f-grams get 16 bits per key, up to 48 M f-grams 8 bits per key (~6 % false positives:
// a 10 M-f-gram filter is 20 MB and still lives in the 126 MB L2 next to the streamed rows), larger ones none.
// ---------------------------------------------------------------------------------------------
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

__device__ __forceinline__ int32_t probe_any(const IndexView &ix, uint64_t h, const int32_t (&key)[7]) {
    if (!filter_pass(ix, h)) return -1;
    return ix.compact == kSlotCompact16 ? probe16(ix, h, key) : ix.compact == kSlotCompact20 ? probe20(ix, h, key) : probe(ix, h, key);
}

// ---------------------------------------------------------------------------------------------
// vector memory helpers
// ---------------------------------------------------------------------------------------------
// L2 evict-first policy for everything that is touched once (cache rows, fallback rows, the output):
// keeps the 126 MB L2 for the index slots.
__device__ __forceinline__ uint64_t policy_evict_first() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ uint64_t policy_evict_last() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ uint4 ldg_stream_16(const void *p, uint64_t pol) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.b32 {%0,%1,%2,%3}, [%4], %5;"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p), "l"(pol));
    return r;
}
__device__ __forceinline__ uint2 ldg_stream_8(const void *p, uint64_t pol) {
    uint2 r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v2.b32 {%0,%1}, [%2], %3;" : "=r"(r.x), "=r"(r.y) : "l"(p), "l"(pol));
    return r;
}
__device__ __forceinline__ uint32_t ldg_stream_4(const void *p, uint64_t pol) {
    uint32_t r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.b32 %0, [%1], %2;" : "=r"(r) : "l"(p), "l"(pol));
    return r;
}
__device__ __forceinline__ void stg_stream_16(void *p, uint4 v, uint64_t pol) {
    asm volatile("st.global.L1::no_allocate.L2::cache_hint.v4.b32 [%0], {%1,%2,%3,%4}, %5;" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w),
                 "l"(pol)
                 : "memory");
}

// streaming read of data touched once (cache rows, fallback rows): no L1 allocation
__device__ __forceinline__ uint4 ldg_stream_16(const void *p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.b32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}
__device__ __forceinline__ uint2 ldg_stream_8(const void *p) {
    uint2 r;
    asm volatile("ld.global.nc.L1::no_allocate.v2.b32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p));
    return r;
}
__device__ __forceinline__ uint32_t ldg_stream_4(const void *p) {
    uint32_t r;
    asm volatile("ld.global.nc.L1::no_allocate.b32 %0, [%1];" : "=r"(r) : "l"(p));
    return r;
}
// write-once output: streaming (evict-first) store
__device__ __forceinline__ void stg_stream_16(void *p, uint4 v) {
    asm volatile("st.global.cs.v4.b32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

// ---------------------------------------------------------------------------------------------
// mbarrier (shared-memory transaction barrier) primitives, used as plain arrive/wait barriers between
// the matcher warp and the gather warps of a CTA
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.release.cta.shared::cta.b64 st, [%0];\n\t}" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.acquire.cta.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t"
        "}" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}

// one arrival that also announces `tx_bytes` of asynchronous (bulk-copy) traffic for this phase
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, uint32_t tx_bytes) {
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.expect_tx.release.cta.shared::cta.b64 st, [%0], %1;\n\t}" ::"r"(smem_u32(bar)),
                 "r"(tx_bytes)
                 : "memory");
}
// TMA 1-D bulk copy global -> shared (UBLKCP); completion is signalled on `bar` as `bytes` of tx.
// dst, src 16-byte aligned, bytes a multiple of 16.
__device__ __forceinline__ void bulk_g2s(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar, uint64_t pol) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)), "l"(pol)
                 : "memory");
}

#endif  // __CUDACC__

}  // namespace scone
