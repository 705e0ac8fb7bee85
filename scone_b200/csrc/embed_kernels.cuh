// embed_kernels.cuh -- the fused hot path: longest-match lookup + cache-row gather + dequant + fallback,
// one kernel, output written once in the transformer's inputs_embeds layout.
//
// Takes over, per position, get_token_f_grams + f_gram_to_id + get_embeddings + the engine's
// assemble loop + the wte fallback of the reference (scone/tokenization/n_gram_extractor.py:106-126,
// scone/inference/embedding_cache.py:149-181, scone/inference/engine.py:235-266,
// scone/models/language_model.py:239-243), with Algorithm-2 (replace-or-fallback) semantics.
//
// Shape of the kernels (HBM-bound gather, no tensor cores):
//   * persistent CTAs (a multiple of the 148 SMs), warp-specialised into NM MATCHER warps and NG GATHER warps.
//   * a matcher walks every NM-th tile of its CTA (a tile = the G = 32/P consecutive positions one warp can match
//     at once, match.cuh), resolves the f-gram ids, writes fgram_id / match_len, and pushes (row id, fallback token)
//     into a small shared-memory ring guarded by mbarriers.  Matchers run ahead of the gather warps, so the dependent
//     chain ids -> hash -> slot -> (re-probe) is off the streaming warps' critical path.
//   * embed_bulk_kernel (default): the matcher also issues ONE TMA bulk copy (cp.async.bulk, global -> shared) per
//     position -- the table row on a hit, the fallback row on a miss -- into the tile's ring slot; the slot's mbarrier
//     completes when the bytes have landed.  Loads in flight are bounded by shared memory, not registers.  Gather warps
//     read the row from shared memory, dequantise, and write 128-bit vectors.
//   * embed_kernel (rows too wide for a ring): gather warps load the row themselves with 128-bit
//     ld.global.nc.L1::no_allocate, U 256-element steps in flight per lane.
//   * everything streamed (rows, fallback rows, output) carries an L2 evict-first policy, index slots evict-last.
//   * every gather warp waits for and releases every tile, in order: with parity-only mbarriers no waiter may be more
//     than one phase away from the barrier's current phase.
//   * extra rows per position (fused position add, additive combine) go through the three-role pipeline of
//     embed_pipe.cuh, or through embed_kernel where rows are too wide for a ring; embed_plan.h picks the kernel.
//
// This header is compiled once per (table format, output type) by embed_inst.cu; embed.cu holds the plan and the C ABI.
#pragma once
#include "embed_plan.h"
#include "match.cuh"
#include "row_format.cuh"

#include <utility>

namespace scone {

struct EmbedParams {
    IndexView ix;
    const int32_t *fgram_in;  // not NULL: ids already resolved, the matcher only forwards them
    const uint8_t *rows;
    const uint8_t *const *shard_rows;  // world > 1: peer-mapped shard base pointers (device array), row r on shard r % world
    int64_t row_stride;
    int64_t num_rows;
    const uint8_t *base;  // [V, D] 16-bit
    int64_t V;
    const uint8_t *pos;  // [>= L, D] 16-bit or NULL
    const int64_t *ids;
    int64_t T, L;
    uint8_t *out;
    int32_t *out_id;
    uint8_t *out_len;
    uint32_t *status;
    int64_t num_tiles;
    int32_t D;
    int32_t scale_off;
    int32_t group_shift;  // log2(group / 8): chunk index >> group_shift = group index (INT4)
    int32_t world;        // 1 = the whole table is at `rows`
    int32_t additive;     // 1 = reference-code combine: base row + table row on a hit (language_model.py:239-243)
    int32_t stagger_ns;   // matcher warp w starts its first probes w * stagger_ns later (0 = together)
    uint32_t flags;       // SCONE_EMBED_* of scone_embed_opts_t
};

// address of table row `fid`: local, or on the peer that owns it (NVLink)
__device__ __forceinline__ const uint8_t *row_ptr(const EmbedParams &p, int32_t fid) {
    if (p.world == 1) return p.rows + (int64_t)fid * p.row_stride;
    const int32_t w = p.world < 0 ? -p.world : p.world;  // negative: sharded, read through the pointer table
    const int32_t owner = fid % w, local = fid / w;
    const uint8_t *base = reinterpret_cast<const uint8_t *>(__ldg(reinterpret_cast<const unsigned long long *>(p.shard_rows) + owner));
    return base + (int64_t)local * p.row_stride;
}

constexpr int kRing = 16;  // tiles embed_kernel's matchers may run ahead of the gather warps

// programmatic dependent launch: block until the grid this one was launched behind has completed and its writes are visible
__device__ __forceinline__ void griddep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// base and position rows are stored in the output type
template <int OUT>
__device__ __forceinline__ void decode16x8(uint4 raw, f32x8 &x) {
    if (OUT == SCONE_OUT_BF16) decode_bf16x8(raw, x);
    else decode_fp16x8(raw, x);
}

// ---- streaming one position -------------------------------------------------------------------------

// A table row's chunk in the output type.  FP16 rows into FP16 output are copied as they are.
template <int QUANT, int OUT>
__device__ __forceinline__ uint4 hit_chunk(const RawChunk &raw) {
    if (QUANT == SCONE_QUANT_FP16 && OUT == SCONE_OUT_FP16) return raw.a;
    f32x8 x;
    decode_chunk<QUANT>(raw, x);
    return pack_chunk<OUT>(x).v[0];
}

// Chunk c of a position that needs more than its table row, in fp32 (the caller packs it to the output type): the table
// row (fid >= 0) or else the fallback row (tok >= 0), both at `src`, or else zeros; + the base row `arow` (additive combine:
// wte(ids) + f-gram row); + the position row `prow`.  The one statement of these fp32 adds and their order for every kernel:
// the output is held bit-exact to the oracle.  Position rows are read through `pmem`.
template <int QUANT, int OUT, class Mem, class PosMem>
__device__ __forceinline__ void combine_chunk(const EmbedParams &p, const Mem &mem, const PosMem &pmem, int32_t fid, int32_t tok,
                                              const uint8_t *src, float rs, const uint8_t *arow, const uint8_t *prow, int c, f32x8 &x) {
    if (fid >= 0) decode_chunk<QUANT>(load_chunk<QUANT>(mem, src, c, p.scale_off, p.group_shift, rs), x);
    else if (tok >= 0) decode16x8<OUT>(mem.v16(src + c * 16), x);
    else zero8(x);
    if (arow) {
        f32x8 y;
        decode16x8<OUT>(mem.v16(arow + c * 16), y);
        add8(x, y);
    }
    if (prow) {
        f32x8 y;
        decode16x8<OUT>(pmem.v16(prow + c * 16), y);
        add8(x, y);
    }
}

// Hit: dequantise table row `fid` into dst.  U 256-element steps in flight per lane.
template <int QUANT, int OUT, int U>
__device__ __forceinline__ void stream_hit(const EmbedParams &p, int32_t fid, uint8_t *__restrict__ dst, int lane, uint64_t pol) {
    const uint8_t *__restrict__ row = row_ptr(p, fid);
    const int nchunks = p.D >> 3;
    const GlobalRowsEvictFirst mem{{}, pol};
    const float rs = row_scale<QUANT>(mem, row, p.scale_off);
    for (int c0 = lane; c0 < nchunks; c0 += 32 * U) {
        RawChunk raw[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int c = c0 + 32 * u;
            if (c < nchunks) raw[u] = load_chunk<QUANT>(mem, row, c, p.scale_off, p.group_shift, rs);
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int c = c0 + 32 * u;
            if (c < nchunks) {
                const uint4 o = hit_chunk<QUANT, OUT>(raw[u]);
                stg_stream_16(dst + c * 16, o, pol);
            }
        }
    }
}

// Miss: the fallback row is already in the output type -> 16 B copy.
template <int U>
__device__ __forceinline__ void stream_miss(const EmbedParams &p, int32_t tok, uint8_t *__restrict__ dst, int lane, uint64_t pol) {
    const uint8_t *__restrict__ row = p.base + (int64_t)tok * p.D * 2;
    const int nchunks = p.D >> 3;
    for (int c0 = lane; c0 < nchunks; c0 += 32 * U) {
        uint4 raw[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int c = c0 + 32 * u;
            if (c < nchunks) raw[u] = ldg_stream_16(row + c * 16, pol);
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int c = c0 + 32 * u;
            if (c < nchunks) stg_stream_16(dst + c * 16, raw[u], pol);
        }
    }
}

// Everything else (position add, out-of-range token): correctness path, not tuned.
template <int QUANT, int OUT>
__device__ __noinline__ void stream_general(const EmbedParams &p, int32_t fid, int32_t tok, int64_t t, uint8_t *__restrict__ dst,
                                            int lane) {
    const int nchunks = p.D >> 3;
    const GlobalRows mem;
    const uint8_t *src = fid >= 0 ? row_ptr(p, fid) : tok >= 0 ? p.base + (int64_t)tok * p.D * 2 : nullptr;
    const float rs = fid >= 0 ? row_scale<QUANT>(mem, src, p.scale_off) : 1.0f;
    const uint8_t *arow = (p.additive && fid >= 0 && tok >= 0) ? p.base + (int64_t)tok * p.D * 2 : nullptr;
    const uint8_t *prow = p.pos ? p.pos + pos_in_row(t, p.L, p.T) * p.D * 2 : nullptr;
    for (int c = lane; c < nchunks; c += 32) {
        f32x8 x;
        combine_chunk<QUANT, OUT>(p, mem, GlobalRowsCached{}, fid, tok, src, rs, arow, prow, c, x);
        stg_stream_16(dst + c * 16, pack_chunk<OUT>(x).v[0]);
    }
}

// ---- the matchers' resolve step ------------------------------------------------------------------------

struct Resolved {
    int32_t fid;  // table row, -1 = miss, -2 = resolved id outside the table (zero row + status)
    int32_t tok;  // token whose base row the position needs, or -1
    int32_t len;  // match length (matching only)
};

// Position lane / P of tile `tile`: the given f-gram id, or the longest match over the token window `wtok`, which is
// replaced by the window of the matcher's next tile `ntile` (requested before the dependent probe chain of this one).
// A miss needs its base row as the fallback, and so does a hit under the additive combine (`add`).
template <int P>
__device__ __forceinline__ Resolved resolve_position(const EmbedParams &p, bool add, int64_t tile, int64_t ntile, int lane, int back,
                                                     int32_t &wtok) {
    constexpr int G = 32 / P;
    const int64_t i = tile * G + lane / P;
    Resolved r{-1, -1, 0};
    if (p.fgram_in) {
        if (i < p.T) {
            r.fid = __ldg(p.fgram_in + i);
            if (r.fid >= p.num_rows) r.fid = -2;  // caller error: zero row + status
            if (r.fid == -1 || (add && r.fid >= 0)) {
                const int64_t t64 = __ldg(p.ids + i);
                if (t64 >= 0 && t64 < p.V) r.tok = (int32_t)t64;
            }
        }
    } else {
        int32_t ntok = -1;
        if (ntile < p.num_tiles) ntok = load_window_token<P>(p.ids, p.T, ntile * G, lane, back);
        const WindowMatch m = match_window<P>(p.ix, wtok, p.T, p.L, tile * G, lane, back);
        r.fid = m.fid;
        r.len = m.len;
        r.tok = own_token<P>(wtok, lane, back);
        if ((int64_t)r.tok >= p.V) r.tok = -1;
        wtok = ntok;
        if (r.fid != -1 && !(add && r.fid >= 0)) r.tok = -1;
    }
    return r;
}

// ---- the kernel --------------------------------------------------------------------------------------

template <int QUANT, int OUT, int P, int U, int NM, int NG, int MINB>
__global__ void __launch_bounds__(32 * (NM + NG), MINB) embed_kernel(const EmbedParams p) {
    constexpr int G = 32 / P;
    static_assert(kRing >= NM, "ring must hold the tiles all matchers have in flight");
    constexpr int R = kRing / NM * NM;  // slot ownership: a ring slot is only ever filled by one matcher
    __shared__ __align__(8) uint64_t full_bar[kRing];
    __shared__ __align__(8) uint64_t empty_bar[kRing];
    __shared__ int2 ring[kRing][G];  // (row id or <0, fallback token or -1)

    // Programmatic dependent launch: let the next kernel in the stream start being scheduled now; its own
    // griddepcontrol.wait (below) still orders it after everything this grid writes.
    asm volatile("griddepcontrol.launch_dependents;");
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) {
#pragma unroll
        for (int q = 0; q < kRing; ++q) {
            mbar_init(&full_bar[q], 1);
            mbar_init(&empty_bar[q], NG);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    // everything above overlapped the previous kernel's tail; nothing below may run before it has completed
    asm volatile("griddepcontrol.wait;" ::: "memory");

    if (warp < NM) {
        // ===== matcher warps: resolve the CTA's tiles round-robin, running ahead of the gather warps =====
        const int j = lane / P;
        const int back = p.ix.max_n - 1;
        int64_t it = warp;
        int64_t tile = blockIdx.x + it * gridDim.x;
        int32_t wtok = -1;
        if (!p.fgram_in && tile < p.num_tiles) wtok = load_window_token<P>(p.ids, p.T, tile * G, lane, back);
        for (; tile < p.num_tiles; it += NM, tile += (int64_t)NM * gridDim.x) {
            const int q = (int)(it % R);
            const int64_t i = tile * G + j;
            const Resolved r = resolve_position<P>(p, p.additive != 0, tile, tile + (int64_t)NM * gridDim.x, lane, back, wtok);
            if (!p.fgram_in && (lane % P) == 0 && i < p.T) {
                if (p.out_id) p.out_id[i] = r.fid;
                if (p.out_len) p.out_len[i] = (uint8_t)r.len;
            }
            mbar_wait(&empty_bar[q], (uint32_t)(((it / R) & 1) ^ 1));
            // lane 0 publishes the whole tile and then arrives: one producer thread per phase
#pragma unroll
            for (int g = 0; g < G; ++g) {
                const int32_t f = __shfl_sync(0xFFFFFFFFu, r.fid, g * P);
                const int32_t k2 = __shfl_sync(0xFFFFFFFFu, r.tok, g * P);
                if (lane == 0) ring[q][g] = make_int2(f, k2);
            }
            if (lane == 0) mbar_arrive(&full_bar[q]);
        }
    } else {
        // ===== gather warps: walk the CTA's tiles in order, stream the positions they own =====
        // Position s = itl * G + j of the CTA's sequence belongs to gather warp s % NG.  EVERY gather warp waits
        // for and releases EVERY tile (even one in which it owns nothing): with parity-only mbarriers this is
        // what guarantees that no waiter is ever more than one phase away from the barrier's current phase.
        bool flagged = false;
        const bool general = p.pos != nullptr || p.additive;
        const uint64_t pol = policy_evict_first();
        const int w = warp - NM;
        int64_t itl = 0;
        for (int64_t tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++itl) {
            const int q = (int)(itl % R);
            mbar_wait(&full_bar[q], (uint32_t)((itl / R) & 1));
            const int first = (int)(((int64_t)w - (itl * G) % NG + NG) % NG);
            for (int j = first; j < G; j += NG) {
                const int2 e = ring[q][j];
                const int64_t t = tile * G + j;
                if (t < p.T) {
                    uint8_t *dst = p.out + t * p.D * 2;
                    if (general || (e.x < 0 && e.y < 0)) {
                        stream_general<QUANT, OUT>(p, e.x, e.y, t, dst, lane);
                        flagged |= e.y < 0 && (e.x < 0 || p.additive);
                    } else if (e.x >= 0) {
                        stream_hit<QUANT, OUT, U>(p, e.x, dst, lane, pol);
                    } else {
                        stream_miss<U>(p, e.y, dst, lane, pol);
                    }
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty_bar[q]);
        }
        if (flagged && p.status && lane == 0) atomicOr(p.status, SCONE_STATUS_TOKEN_OOR);
    }
}

// ---- variant B: rows land in shared memory through TMA bulk copies ---------------------------------------
//
// Same roles, but the matcher that resolved a tile also issues one cp.async.bulk (global -> shared, 1-D) per
// position into the tile's ring slot; the slot's mbarrier completes when the matcher has arrived AND all row
// bytes have landed.  Loads in flight are then bounded by shared memory (tens of KB per CTA) instead of by the
// gather warps' registers, and the gather warps only touch shared memory and issue the output stores.

template <int QUANT, int OUT>
__device__ __forceinline__ void stream_from_smem(const EmbedParams &p, const uint8_t *srow, const uint8_t *arow, const uint8_t *prow,
                                                 int32_t fid, int32_t tok, uint8_t *__restrict__ dst, int lane, uint64_t pol) {
    const int nchunks = p.D >> 3;  // arow / prow: base row to add to a hit / position-embedding row, in shared memory, or NULL
    const SharedRows mem;
    if (fid >= 0 && !prow && !arow) {
        const float rs = row_scale<QUANT>(mem, srow, p.scale_off);
#pragma unroll 4
        for (int c = lane; c < nchunks; c += 32) {
            const uint4 o = hit_chunk<QUANT, OUT>(load_chunk<QUANT>(mem, srow, c, p.scale_off, p.group_shift, rs));
            stg_stream_16(dst + c * 16, o, pol);
        }
    } else if (fid < 0 && tok >= 0 && !prow) {
#pragma unroll 4
        for (int c = lane; c < nchunks; c += 32) stg_stream_16(dst + c * 16, *reinterpret_cast<const uint4 *>(srow + c * 16), pol);
    } else {
        // base-row add, position add (the matcher staged those rows next to the table row) / zero row
        float rs = 1.0f;
        if (fid >= 0) rs = row_scale<QUANT>(mem, srow, p.scale_off);
        for (int c0 = lane; c0 < nchunks; c0 += 128) {
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int c = c0 + 32 * u;
                if (c >= nchunks) continue;
                f32x8 x;
                combine_chunk<QUANT, OUT>(p, mem, mem, fid, tok, srow, rs, arow, prow, c, x);
                stg_stream_16(dst + c * 16, pack_chunk<OUT>(x).v[0], pol);
            }
        }
    }
}

// The plain path only: no position rows, no additive combine (those run on embed_pipe_kernel, DESIGN section 4.2).
template <int QUANT, int OUT, int P, int NM, int NG, int MINB>
__global__ void __launch_bounds__(32 * (NM + NG), MINB) embed_bulk_kernel(const EmbedParams p, const BulkLayout lay) {
    constexpr int G = 32 / P;
    extern __shared__ __align__(128) uint8_t smem[];
    uint64_t *full_bar = reinterpret_cast<uint64_t *>(smem);
    uint64_t *empty_bar = full_bar + kMaxRing;
    int2 *ring = reinterpret_cast<int2 *>(empty_bar + kMaxRing);  // [ring][G]
    uint8_t *rows_smem = smem + bulk_header_bytes(G);
    const int R = lay.ring;

    asm volatile("griddepcontrol.launch_dependents;");
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) {
        for (int q = 0; q < R; ++q) {
            mbar_init(&full_bar[q], 1);
            mbar_init(&empty_bar[q], NG);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    // Everything above overlapped the previous kernel's tail.  By default nothing below may run before that kernel has
    // completed.  With SCONE_EMBED_INPUTS_STABLE the caller vouches that no INPUT of this call (ids, index, table rows,
    // base / position rows) is written by the kernel that precedes it in the stream: matching and the row copies into
    // shared memory then start at once -- the whole dependent chain ids -> slot -> row runs under the previous kernel's
    // tail -- and only the first WRITE to global memory (fgram_id / match_len here, the embeddings in the gather warps)
    // waits for the previous grid.
    const bool early = (p.flags & SCONE_EMBED_INPUTS_STABLE) != 0;
    bool waited = !early;
    if (!early) griddep_wait();

    if (warp < NM) {
        const int j = lane / P;
        const int back = p.ix.max_n - 1;
        const uint64_t pol = policy_evict_first();
        int64_t it = warp;
        int64_t tile = blockIdx.x + it * gridDim.x;
        int32_t wtok = -1;
        if (!p.fgram_in && tile < p.num_tiles) wtok = load_window_token<P>(p.ids, p.T, tile * G, lane, back);
        // The first probes of all matchers of all CTAs would hit the index as one burst of random 64-byte reads; spreading
        // them lets the first tiles resolve (and their rows start to flow) before the burst has drained.
        if (!p.fgram_in) {
            const unsigned wait_ns = (unsigned)(warp * p.stagger_ns);
            if (wait_ns) __nanosleep(wait_ns);
        }
        for (; tile < p.num_tiles; it += NM, tile += (int64_t)NM * gridDim.x) {
            const int q = (int)(it % R);
            const int64_t i = tile * G + j;
            const Resolved r = resolve_position<P>(p, false, tile, tile + (int64_t)NM * gridDim.x, lane, back, wtok);
            // source of this position's bytes
            const bool owner = (lane % P) == 0 && i < p.T;
            const uint8_t *src = nullptr;
            uint32_t bytes = 0;
            if (owner) {
                if (r.fid >= 0) {
                    src = row_ptr(p, r.fid);
                    bytes = (uint32_t)p.row_stride;
                } else if (r.tok >= 0) {
                    src = p.base + (int64_t)r.tok * p.D * 2;
                    bytes = (uint32_t)p.D * 2u;
                }
            }
            uint32_t total = bytes;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) total += __shfl_xor_sync(0xFFFFFFFFu, total, o);
            mbar_wait(&empty_bar[q], (uint32_t)(((it / R) & 1) ^ 1));
            // lane 0 publishes the whole tile and then arrives: one producer thread per phase
#pragma unroll
            for (int g = 0; g < G; ++g) {
                const int32_t f = __shfl_sync(0xFFFFFFFFu, r.fid, g * P);
                const int32_t k2 = __shfl_sync(0xFFFFFFFFu, r.tok, g * P);
                if (lane == 0) ring[q * G + g] = make_int2(f, k2);
            }
            if (lane == 0) mbar_arrive_expect_tx(&full_bar[q], total);
            __syncwarp();
            if (bytes) bulk_g2s(rows_smem + (size_t)(q * G + j) * lay.slot_bytes, src, bytes, &full_bar[q], pol);
            // the match result is this warp's only global write: after the previous grid (see `early` above)
            if (!waited) {
                griddep_wait();
                waited = true;
            }
            if (!p.fgram_in && owner) {
                if (p.out_id) p.out_id[i] = r.fid;
                if (p.out_len) p.out_len[i] = (uint8_t)r.len;
            }
        }
    } else {
        // every gather warp waits for and releases every tile, in order (see embed_kernel)
        bool flagged = false;
        const uint64_t pol = policy_evict_first();
        const int w = warp - NM;
        int64_t itl = 0;
        for (int64_t tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++itl) {
            const int q = (int)(itl % R);
            mbar_wait(&full_bar[q], (uint32_t)((itl / R) & 1));
            if (!waited) {  // rows are staged; the stores below are the first thing that must follow the previous grid
                griddep_wait();
                waited = true;
            }
            const int first = (int)(((int64_t)w - (itl * G) % NG + NG) % NG);
            for (int j = first; j < G; j += NG) {
                const int2 e = ring[q * G + j];
                const int64_t t = tile * G + j;
                if (t < p.T) {
                    stream_from_smem<QUANT, OUT>(p, rows_smem + (size_t)(q * G + j) * lay.slot_bytes, nullptr, nullptr, e.x, e.y,
                                                 p.out + t * p.D * 2, lane, pol);
                    flagged |= e.y < 0 && e.x < 0;
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty_bar[q]);
        }
        if (flagged && p.status && lane == 0) atomicOr(p.status, SCONE_STATUS_TOKEN_OOR);
    }
}


}  // namespace scone
#include "embed_pipe.cuh"
namespace scone {

// Launches kern(p, lay...) as planned: a persistent grid over the call's tiles, programmatic stream serialization (PDL).
// Back-to-back steps overlap this kernel's launch and prologue (barrier init) with the previous kernel's tail; its
// griddepcontrol.wait still orders everything it reads or writes after the previous grid.  Same-box A/B on B200: config 1
// -8 %, config 2 -1.6 %, config 3 unchanged.
template <auto kern, typename... Layout>
static int launch_resident(const EmbedPlan &pl, EmbedParams &p, cudaStream_t stream, Layout... lay) {
    static int configured[64] = {0};  // per device: the attribute lives in the device's context
    int dev = 0;
    SCONE_CUDA(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64 || configured[dev] < pl.smem_bytes) {
        SCONE_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, pl.smem_bytes));
        if (dev >= 0 && dev < 64) configured[dev] = pl.smem_bytes;
    }
    p.num_tiles = pl.num_tiles;
    p.stagger_ns = pl.stagger_ns;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)pl.grid);
    cfg.blockDim = dim3(pl.threads);
    cfg.dynamicSmemBytes = (size_t)pl.smem_bytes;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    SCONE_CUDA(cudaLaunchKernelEx(&cfg, kern, p, lay...));
    return SCONE_OK;
}

template <int QUANT, int OUT, ShapeId S, int P, bool ADD>
static int launch_shape(const EmbedPlan &pl, EmbedParams &p, cudaStream_t stream) {
    constexpr ShapeRow s = kShapes[S];
    if constexpr (s.family == kBulk) {
        return launch_resident<embed_bulk_kernel<QUANT, OUT, P, s.nm, s.ng, s.minb>>(pl, p, stream, pl.bulk);
    } else if constexpr (s.family == kPipe) {
        static_assert(s.nl <= 32 / P, "a loader without a position");
        return launch_resident<embed_pipe_kernel<QUANT, OUT, P, s.nm, s.nl, s.ng, s.minb, ADD>>(pl, p, stream, pl.pipe);
    } else {
        return launch_resident<embed_kernel<QUANT, OUT, P, 4, s.nm, s.ng, s.minb>>(pl, p, stream);  // reads p.additive
    }
}

// K = (shape row, log2 P, ADD): launches the plan if it is that combination and kShapes lists it (nothing else is compiled)
template <int QUANT, int OUT, int K>
static bool launch_if_planned(const EmbedPlan &pl, EmbedParams &p, cudaStream_t stream, int &rc) {
    constexpr ShapeId S = ShapeId(K / 8);
    constexpr int P = 1 << (K / 2 % 4);
    constexpr bool ADD = K % 2;
    if constexpr (((ADD ? kShapes[S].add : kShapes[S].plain) & P) != 0) {
        if (pl.row == S && pl.P == P && pl.add == ADD) {
            rc = launch_shape<QUANT, OUT, S, P, ADD>(pl, p, stream);
            return true;
        }
    }
    return false;
}

template <int QUANT, int OUT, int... K>
static int launch_planned(const EmbedPlan &pl, EmbedParams &p, cudaStream_t stream, std::integer_sequence<int, K...>) {
    int rc = SCONE_OK;
    if (!(launch_if_planned<QUANT, OUT, K>(pl, p, stream, rc) || ...)) {
        set_error("scone_embed: no kernel compiled for shape %d, P %d, additive %d", (int)pl.row, pl.P, (int)pl.add);
        return SCONE_E_INVALID;
    }
    return rc;
}

// one per (table format, output type): embed_inst.cu
template <int QUANT, int OUT>
int launch_plan(const EmbedPlan &pl, EmbedParams &p, cudaStream_t stream) {
    return launch_planned<QUANT, OUT>(pl, p, stream, std::make_integer_sequence<int, kNumShapes * 8>{});
}

}  // namespace scone
