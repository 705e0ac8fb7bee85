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
