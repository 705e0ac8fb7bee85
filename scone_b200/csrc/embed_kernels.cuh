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
//   * optional extra rows per position ride in the same ring slot: the position-embedding row (fused wpe add) and, in the
//     additive combine (template parameter ADD), the base row of a hit.
//
// This header is compiled once per (table format, output type) by embed_inst.cu; embed.cu holds dispatch and the C ABI.
#pragma once
#include "common.cuh"
#include "match.cuh"

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

// row bytes holding 8 consecutive elements of a stored row
template <int QUANT>
__host__ __device__ constexpr int chunk_bytes() {
    return QUANT == SCONE_QUANT_FP32 ? 32 : QUANT == SCONE_QUANT_FP16 ? 16 : QUANT == SCONE_QUANT_INT8 ? 8 : 4;
}

// address of table row `fid`: local, or on the peer that owns it (NVLink)
__device__ __forceinline__ const uint8_t *row_ptr(const EmbedParams &p, int32_t fid) {
    if (p.world == 1) return p.rows + (int64_t)fid * p.row_stride;
    const int32_t w = p.world < 0 ? -p.world : p.world;  // negative: sharded, read through the pointer table
    const int32_t owner = fid % w, local = fid / w;
    const uint8_t *base = reinterpret_cast<const uint8_t *>(__ldg(reinterpret_cast<const unsigned long long *>(p.shard_rows) + owner));
    return base + (int64_t)local * p.row_stride;
}

constexpr int kRing = 16;  // tiles the matchers may run ahead of the gather warps
constexpr uint32_t kEmbedPipe = 1u << 31;  // EmbedParams::flags, internal: use embed_pipe_kernel instead of embed_bulk_kernel

// programmatic dependent launch: block until the grid this one was launched behind has completed and its writes are visible
__device__ __forceinline__ void griddep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

template <int OUT>
__device__ __forceinline__ void decode16x8(uint4 raw, f32x8 &x) {
    if (OUT == SCONE_OUT_BF16) decode_bf16x8(raw, x);
    else decode_fp16x8(raw, x);
}
template <int OUT>
__device__ __forceinline__ uint4 pack16x8(const f32x8 &x) {
    return OUT == SCONE_OUT_BF16 ? pack_bf16x8(x) : pack_fp16x8(x);
}

// ---- streaming one position -------------------------------------------------------------------------

// Hit: dequantise table row `fid` into dst.  U 256-element steps in flight per lane.
template <int QUANT, int OUT, int U>
__device__ __forceinline__ void stream_hit(const EmbedParams &p, int32_t fid, uint8_t *__restrict__ dst, int lane, uint64_t pol) {
    const uint8_t *__restrict__ row = row_ptr(p, fid);
    const int nchunks = p.D >> 3;
    float rs = 1.0f;
    if (QUANT == SCONE_QUANT_INT8) rs = __ldg(reinterpret_cast<const float *>(row + p.scale_off));
    for (int c0 = lane; c0 < nchunks; c0 += 32 * U) {
        uint4 raw[U], rawb[U];  // rawb: second half of an fp32 chunk
        float sc[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int c = c0 + 32 * u;
            sc[u] = rs;
            if (c < nchunks) {
                if (QUANT == SCONE_QUANT_FP32) {
                    raw[u] = ldg_stream_16(row + c * 32, pol);
                    rawb[u] = ldg_stream_16(row + c * 32 + 16, pol);
                } else if (QUANT == SCONE_QUANT_FP16) {
                    raw[u] = ldg_stream_16(row + c * 16, pol);
                } else if (QUANT == SCONE_QUANT_INT8) {
                    const uint2 v = ldg_stream_8(row + c * 8, pol);
                    raw[u].x = v.x;
                    raw[u].y = v.y;
                } else {
                    raw[u].x = ldg_stream_4(row + c * 4, pol);
                    sc[u] = __half2float(__ldg(reinterpret_cast<const __half *>(row + p.scale_off) + (c >> p.group_shift)));
                }
            }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int c = c0 + 32 * u;
            if (c < nchunks) {
                uint4 o;
                if (QUANT == SCONE_QUANT_FP16 && OUT == SCONE_OUT_FP16) {
                    o = raw[u];
                } else {
                    f32x8 x;
                    if (QUANT == SCONE_QUANT_FP32) decode_fp32x8(raw[u], rawb[u], x);
                    else if (QUANT == SCONE_QUANT_FP16) decode_fp16x8(raw[u], x);
                    else if (QUANT == SCONE_QUANT_INT8) decode_int8x8(make_uint2(raw[u].x, raw[u].y), sc[u], x);
                    else decode_int4x8(raw[u].x, sc[u], x);
                    o = pack16x8<OUT>(x);
                }
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
    const uint8_t *row = fid >= 0 ? row_ptr(p, fid) : nullptr;
    const uint8_t *brow = (fid < 0 && tok >= 0) ? p.base + (int64_t)tok * p.D * 2 : nullptr;
    const uint8_t *arow = (p.additive && fid >= 0 && tok >= 0) ? p.base + (int64_t)tok * p.D * 2 : nullptr;
    const uint8_t *prow = p.pos ? p.pos + pos_in_row(t, p.L, p.T) * p.D * 2 : nullptr;
    for (int c = lane; c < nchunks; c += 32) {
        f32x8 x;
        if (row) {
            if (QUANT == SCONE_QUANT_FP32) {
                decode_fp32x8(ldg_stream_16(row + c * 32), ldg_stream_16(row + c * 32 + 16), x);
            } else if (QUANT == SCONE_QUANT_FP16) {
                decode_fp16x8(ldg_stream_16(row + c * 16), x);
            } else if (QUANT == SCONE_QUANT_INT8) {
                decode_int8x8(ldg_stream_8(row + c * 8), __ldg(reinterpret_cast<const float *>(row + p.scale_off)), x);
            } else {
                const __half hs = __ldg(reinterpret_cast<const __half *>(row + p.scale_off) + (c >> p.group_shift));
                decode_int4x8(ldg_stream_4(row + c * 4), __half2float(hs), x);
            }
        } else if (brow) {
            decode16x8<OUT>(ldg_stream_16(brow + c * 16), x);
        } else {
            zero8(x);
        }
        if (arow) {  // wte(ids) + f-gram row
            f32x8 y;
            decode16x8<OUT>(ldg_stream_16(arow + c * 16), y);
            add8(x, y);
        }
        if (prow) {
            f32x8 y;
            decode16x8<OUT>(__ldg(reinterpret_cast<const uint4 *>(prow + c * 16)), y);
            add8(x, y);
        }
        stg_stream_16(dst + c * 16, pack16x8<OUT>(x));
    }
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
            const int64_t base = tile * G;
            const int64_t i = base + j;
            // the ids of this warp's NEXT tile are requested before the dependent probe chain of this one
            const int64_t ntile = tile + (int64_t)NM * gridDim.x;
            int32_t ntok = -1;
            int32_t fid = -1, tok = -1;
            if (p.fgram_in) {
                if (i < p.T) {
                    fid = __ldg(p.fgram_in + i);
                    if (fid >= p.num_rows) fid = -2;  // caller error: zero row + status
                    if (fid == -1 || (p.additive && fid >= 0)) {
                        const int64_t t64 = __ldg(p.ids + i);
                        if (t64 >= 0 && t64 < p.V) tok = (int32_t)t64;
                    }
                }
            } else {
                if (ntile < p.num_tiles) ntok = load_window_token<P>(p.ids, p.T, ntile * G, lane, back);
                const WindowMatch m = match_window<P>(p.ix, wtok, p.T, p.L, base, lane, back);
                fid = m.fid;
                tok = own_token<P>(wtok, lane, back);
                if ((int64_t)tok >= p.V) tok = -1;
                if ((lane % P) == 0 && i < p.T) {
                    if (p.out_id) p.out_id[i] = m.fid;
                    if (p.out_len) p.out_len[i] = (uint8_t)m.len;
                }
                wtok = ntok;
            }
            mbar_wait(&empty_bar[q], (uint32_t)(((it / R) & 1) ^ 1));
            // lane 0 publishes the whole tile and then arrives: one producer thread per phase
            const int32_t tk = (fid == -1 || (p.additive && fid >= 0)) ? tok : -1;  // the base row is needed
#pragma unroll
            for (int g = 0; g < G; ++g) {
                const int32_t f = __shfl_sync(0xFFFFFFFFu, fid, g * P);
                const int32_t k2 = __shfl_sync(0xFFFFFFFFu, tk, g * P);
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

struct BulkLayout {
    int ring;        // ring slots (tiles in flight per CTA)
    int slot_bytes;  // bytes reserved per position: the row (>= max(row_stride, 2 D)) [+ base row] [+ position row], multiple of 128
    int pos_off;     // offset of the position-embedding row inside a position's slot, 0 = no position add
    int add_off;     // offset of the base row staged next to a HIT's table row (additive combine), 0 = replace mode
    int smem_bytes;  // dynamic shared memory per CTA
};

// 8 elements (chunk c) of a table row staged in shared memory -> fp32
template <int QUANT>
__device__ __forceinline__ void decode_smem(const EmbedParams &p, const uint8_t *srow, int c, float rs, f32x8 &x) {
    if (QUANT == SCONE_QUANT_FP32) {
        decode_fp32x8(*reinterpret_cast<const uint4 *>(srow + c * 32), *reinterpret_cast<const uint4 *>(srow + c * 32 + 16), x);
    } else if (QUANT == SCONE_QUANT_FP16) {
        decode_fp16x8(*reinterpret_cast<const uint4 *>(srow + c * 16), x);
    } else if (QUANT == SCONE_QUANT_INT8) {
        decode_int8x8(*reinterpret_cast<const uint2 *>(srow + c * 8), rs, x);
    } else {
        const float sc = __half2float(*(reinterpret_cast<const __half *>(srow + p.scale_off) + (c >> p.group_shift)));
        decode_int4x8(*reinterpret_cast<const uint32_t *>(srow + c * 4), sc, x);
    }
}

template <int QUANT, int OUT>
__device__ __forceinline__ void stream_from_smem(const EmbedParams &p, const uint8_t *srow, const uint8_t *arow, const uint8_t *prow,
                                                 int32_t fid, int32_t tok, uint8_t *__restrict__ dst, int lane, uint64_t pol) {
    const int nchunks = p.D >> 3;  // arow / prow: base row to add to a hit / position-embedding row, in shared memory, or NULL
    if (fid >= 0 && !prow && !arow) {
        float rs = 1.0f;
        if (QUANT == SCONE_QUANT_INT8) rs = *reinterpret_cast<const float *>(srow + p.scale_off);
#pragma unroll 4
        for (int c = lane; c < nchunks; c += 32) {
            uint4 o;
            if (QUANT == SCONE_QUANT_FP16 && OUT == SCONE_OUT_FP16) {
                o = *reinterpret_cast<const uint4 *>(srow + c * 16);
            } else {
                f32x8 x;
                decode_smem<QUANT>(p, srow, c, rs, x);
                o = pack16x8<OUT>(x);
            }
            stg_stream_16(dst + c * 16, o, pol);
        }
    } else if (fid < 0 && tok >= 0 && !prow) {
#pragma unroll 4
        for (int c = lane; c < nchunks; c += 32) stg_stream_16(dst + c * 16, *reinterpret_cast<const uint4 *>(srow + c * 16), pol);
    } else {
        // base-row add, position add (the matcher staged those rows next to the table row) / zero row
        float rs = 1.0f;
        if (QUANT == SCONE_QUANT_INT8 && fid >= 0) rs = *reinterpret_cast<const float *>(srow + p.scale_off);
        for (int c0 = lane; c0 < nchunks; c0 += 128) {
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int c = c0 + 32 * u;
                if (c >= nchunks) continue;
                f32x8 x;
                if (fid >= 0) {
                    decode_smem<QUANT>(p, srow, c, rs, x);
                } else if (tok >= 0) {
                    decode16x8<OUT>(*reinterpret_cast<const uint4 *>(srow + c * 16), x);
                } else {
                    zero8(x);
                }
                if (arow) {  // wte(ids) + f-gram row
                    f32x8 y;
                    decode16x8<OUT>(*reinterpret_cast<const uint4 *>(arow + c * 16), y);
                    add8(x, y);
                }
                if (prow) {
                    f32x8 y;
                    decode16x8<OUT>(*reinterpret_cast<const uint4 *>(prow + c * 16), y);
                    add8(x, y);
                }
                stg_stream_16(dst + c * 16, pack16x8<OUT>(x), pol);
            }
        }
    }
}

constexpr int kMaxRing = 16;
// bytes of barriers + ring metadata in front of the row slots
__host__ __device__ constexpr int bulk_header_bytes(int G) { return (2 * kMaxRing * 8 + kMaxRing * G * 8 + 127) / 128 * 128; }

// ADD (compile time) = the additive combine: measured as a run-time flag it cost the plain path 1-7 % (config 1 6.56 vs
// 6.28 us, config 2 + wpe 57.2 vs 53.1 us, config 3 1017 vs 1006 us), so the plain kernels do not carry it.
template <int QUANT, int OUT, int P, int NM, int NG, int MINB, bool ADD>
__global__ void __launch_bounds__(32 * (NM + NG), MINB) embed_bulk_kernel(const EmbedParams p, const BulkLayout lay) {
    constexpr int G = 32 / P;
    const int add_off = ADD ? lay.add_off : 0;
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
            const int64_t base = tile * G;
            const int64_t i = base + j;
            const int64_t ntile = tile + (int64_t)NM * gridDim.x;
            int32_t ntok = -1;
            int32_t fid = -1, tok = -1, mlen = 0;
            if (p.fgram_in) {
                if (i < p.T) {
                    fid = __ldg(p.fgram_in + i);
                    if (fid >= p.num_rows) fid = -2;
                    if (fid == -1 || (ADD && fid >= 0)) {
                        const int64_t t64 = __ldg(p.ids + i);
                        if (t64 >= 0 && t64 < p.V) tok = (int32_t)t64;
                    }
                }
            } else {
                if (ntile < p.num_tiles) ntok = load_window_token<P>(p.ids, p.T, ntile * G, lane, back);
                const WindowMatch m = match_window<P>(p.ix, wtok, p.T, p.L, base, lane, back);
                fid = m.fid;
                mlen = m.len;
                tok = own_token<P>(wtok, lane, back);
                if ((int64_t)tok >= p.V) tok = -1;
                wtok = ntok;
            }
            if (fid != -1 && !(ADD && fid >= 0)) tok = -1;  // additive: a hit still needs its base row
            // source of this position's bytes
            const bool owner = (lane % P) == 0 && i < p.T;
            const uint8_t *src = nullptr;
            uint32_t bytes = 0;
            if (owner) {
                if (fid >= 0) {
                    src = row_ptr(p, fid);
                    bytes = (uint32_t)p.row_stride;
                } else if (tok >= 0) {
                    src = p.base + (int64_t)tok * p.D * 2;
                    bytes = (uint32_t)p.D * 2u;
                }
            }
            // additive combine: the base row of a hit rides along too (language_model.py:239-243 fused)
            const uint8_t *src3 = nullptr;
            if (add_off && owner && fid >= 0 && tok >= 0) src3 = p.base + (int64_t)tok * p.D * 2;
            // the position-embedding row rides along into the same slot (language_model.py:253-254 fused)
            const uint8_t *src2 = nullptr;
            if (lay.pos_off && owner) src2 = p.pos + pos_in_row(i, p.L, p.T) * p.D * 2;
            uint32_t total = bytes + (src2 ? (uint32_t)p.D * 2u : 0u) + (src3 ? (uint32_t)p.D * 2u : 0u);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) total += __shfl_xor_sync(0xFFFFFFFFu, total, o);
            mbar_wait(&empty_bar[q], (uint32_t)(((it / R) & 1) ^ 1));
            // lane 0 publishes the whole tile and then arrives: one producer thread per phase
#pragma unroll
            for (int g = 0; g < G; ++g) {
                const int32_t f = __shfl_sync(0xFFFFFFFFu, fid, g * P);
                const int32_t k2 = __shfl_sync(0xFFFFFFFFu, tok, g * P);
                if (lane == 0) ring[q * G + g] = make_int2(f, k2);
            }
            if (lane == 0) mbar_arrive_expect_tx(&full_bar[q], total);
            __syncwarp();
            uint8_t *slot = rows_smem + (size_t)(q * G + j) * lay.slot_bytes;
            if (bytes) bulk_g2s(slot, src, bytes, &full_bar[q], pol);
            if (src2) bulk_g2s(slot + lay.pos_off, src2, (uint32_t)p.D * 2u, &full_bar[q], policy_evict_last());
            if (src3) bulk_g2s(slot + add_off, src3, (uint32_t)p.D * 2u, &full_bar[q], pol);
            // the match result is this warp's only global write: after the previous grid (see `early` above)
            if (!waited) {
                griddep_wait();
                waited = true;
            }
            if (!p.fgram_in && owner) {
                if (p.out_id) p.out_id[i] = fid;
                if (p.out_len) p.out_len[i] = (uint8_t)mlen;
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
                    const uint8_t *slot = rows_smem + (size_t)(q * G + j) * lay.slot_bytes;
                    const uint8_t *arow = (add_off && e.x >= 0 && e.y >= 0) ? slot + add_off : nullptr;
                    stream_from_smem<QUANT, OUT>(p, slot, arow, lay.pos_off ? slot + lay.pos_off : nullptr, e.x, e.y, p.out + t * p.D * 2, lane,
                                                 pol);
                    flagged |= e.y < 0 && (e.x < 0 || add_off);
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

static int num_sms() {
    static int n = 0;
    if (n == 0) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
            n = kNumSMsB200;
    }
    return n;
}

// Launches kern(p[, lay]) as a persistent grid over the call's tiles of G positions: at most MINB CTAs per SM, `smem` bytes
// of dynamic shared memory.  Kernels are launched with programmatic stream serialization (PDL): back-to-back steps overlap this kernel's launch
// and prologue (barrier init) with the previous kernel's tail; its griddepcontrol.wait still orders everything it reads
// or writes after the previous grid.  Same-box A/B on B200: config 1 -8 %, config 2 -1.6 %, config 3 unchanged.
template <auto kern, int G, int MINB, typename... Layout>
static int launch_resident(EmbedParams &p, unsigned threads, int smem, cudaStream_t stream, Layout... lay) {
    static int configured[64] = {0};  // per device: the attribute lives in the device's context
    int dev = 0;
    SCONE_CUDA(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64 || configured[dev] < smem) {
        SCONE_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        if (dev >= 0 && dev < 64) configured[dev] = smem;
    }
    p.num_tiles = (p.T + G - 1) / G;
    const int64_t resident = (int64_t)num_sms() * MINB;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)(p.num_tiles < resident ? p.num_tiles : resident));
    cfg.blockDim = dim3(threads);
    cfg.dynamicSmemBytes = (size_t)smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    SCONE_CUDA(cudaLaunchKernelEx(&cfg, kern, p, lay...));
    return SCONE_OK;
}

template <int QUANT, int OUT, int P, int U, int NM, int NG, int MINB>
static int launch_ldg(EmbedParams &p, cudaStream_t stream) {
    return launch_resident<embed_kernel<QUANT, OUT, P, U, NM, NG, MINB>, 32 / P, MINB>(p, 32 * (NM + NG), 0, stream);
}

// Ring geometry for the bulk variant; returns false when rows are too wide for the budget.
// The ring needs at least as many slots as matchers: gather warps release tiles strictly in order, so a matcher that
// has filled tile t - NM knows every tile <= t - NM - ring is consumed; with ring >= NM that covers t - 2 ring, i.e. its
// parity wait on slot t % ring is never more than one phase ahead.
static bool bulk_layout(const EmbedParams &p, int G, int nm, int budget_bytes, BulkLayout &lay) {
    int64_t slot = p.row_stride > 2ll * p.D ? p.row_stride : 2ll * p.D;
    slot = (slot + 127) / 128 * 128;
    lay.pos_off = lay.add_off = 0;
    if (p.additive) {  // room for a hit's base row behind the table row
        lay.add_off = (int)slot;
        slot += (2ll * p.D + 127) / 128 * 128;
    }
    if (p.pos) {  // room for the position-embedding row behind those
        lay.pos_off = (int)slot;
        slot += (2ll * p.D + 127) / 128 * 128;
    }
    const int64_t per_tile = slot * G;
    int ring = (int)((budget_bytes - bulk_header_bytes(G)) / per_tile);
    if (ring > kMaxRing) ring = kMaxRing;
    if (ring < 2 || ring < nm) return false;
    lay.ring = ring;
    lay.slot_bytes = (int)slot;
    lay.smem_bytes = bulk_header_bytes(G) + (int)(per_tile * ring);
    return true;
}

template <int QUANT, int OUT, int P, int NM, int NG, int MINB, bool ADD>
static int launch_bulk(EmbedParams &p, const BulkLayout &lay, cudaStream_t stream) {
    return launch_resident<embed_bulk_kernel<QUANT, OUT, P, NM, NG, MINB, ADD>, 32 / P, MINB>(p, 32 * (NM + NG), lay.smem_bytes, stream, lay);
}

template <int QUANT, int OUT, int P, int NM, int NL, int NG, int MINB, bool ADD>
static int launch_pipe(EmbedParams &p, const PipeLayout &lay, cudaStream_t stream) {
    constexpr int G = 32 / P;
    static_assert(NL <= G, "a loader without a position");
    return launch_resident<embed_pipe_kernel<QUANT, OUT, P, NM, NL, NG, MINB, ADD>, G, MINB>(p, 32 * (NM + NL + NG), lay.smem_bytes, stream, lay);
}

// Kernel selection (measured on B200, profiles/tune_r01.md and tune_r02.md).  Rows that fit a shared-memory ring go through
// one of the two bulk-copy kernels (embed.cu picks: single ring for the plain path, pipeline for extra rows per position and
// for fp32 rows of 2-6 KB); the shape follows the traffic per position.  Single-ring kernel (embed_bulk_kernel):
//   kNarrow6  < 6 KB moved, tiny rows : 6 matcher + 4 gather warps, 3 CTAs/SM, 70 KB ring  (needs >= 6 ring slots)
//   kNarrow4  < 6 KB moved            : 4 matcher + 4 gather warps, 3 CTAs/SM, 70 KB ring  -- matcher-hungry
//   kWide    >= 6 KB moved            : 6 matcher + 12 gather warps, 1 CTA/SM, 200 KB ring -- store-hungry
//   kWide3   wide rows + position row : 3 matcher + 12 gather warps, 1 CTA/SM, 200 KB ring (when six slots do not fit)
//   kWide2   wide rows + base + pos row: 2 matcher + 12 gather warps, 1 CTA/SM, 200 KB ring (two slots are enough)
//   kMid     narrow rows + extra rows : 4 matcher + 8 gather warps, 2 CTAs/SM, 100 KB ring
//   kSmall   anything                 : 2 matcher + 6 gather warps, 3 CTAs/SM, 70 KB ring
//   kLdg     rows too wide for a ring : register-load variant
// Pipeline kernel (embed_pipe_kernel; the ring only needs two full-size tiles), matcher + loader + gather warps:
//   kNarrow6  6 + 1 + 4, 3 CTAs/SM, 70 KB    (config 2 + wpe: 47 us; + base row: 51 us)
//   kNarrow4  5 + 2 + 4, 3 CTAs/SM, 70 KB    (plain path, fp32 rows of 3-4 KB)
//   kMid      4 + 2 + 8, 2 CTAs/SM, 110 KB   (config 2 + base row + wpe: 56 us; fp32 rows of 5-6 KB)
//   kWide*    6 + 4 + 12, 1 CTA/SM, 200 KB   (config 3 modes)
//   kSmall    2 + 1 + 6, 3 CTAs/SM, 70 KB
// A shape that does not fit with P lanes per position is retried with 2P, 4P (fewer positions per tile = smaller ring
// slots) before the next shape is considered.
enum Shape : int { kNarrow6 = 0, kNarrow4 = 1, kWide = 2, kSmall = 3, kLdg = 4, kWide3 = 5, kMid = 6, kWide2 = 7 };
constexpr int kNoFit = 1;

// Matcher start-up stagger (EmbedParams::stagger_ns), narrow shapes only.  Measured on config 2 (profiles/tune_r01.md):
// 400-800 ns per matcher warp is worth 1.5 % with the pre-filter (43.3 -> 42.6 us) and 3 % without it (46.7 -> 45.3 us);
// no effect on the wide shapes; below two tiles per matcher the delay would be exposed instead.
template <int P, int NM, int MINB>
static void set_stagger(EmbedParams &p) {
    constexpr int G = 32 / P;
    if ((p.T + G - 1) / G >= 2ll * NM * MINB * num_sms()) p.stagger_ns = 500;
}

template <int QUANT, int OUT, int P, bool ADD>
static int launch(EmbedParams &p, cudaStream_t stream, int shape) {
    constexpr int G = 32 / P;
    BulkLayout lay;
    if (p.flags & kEmbedPipe) {
        // three-role pipeline (embed_pipe.cuh): tiles keep their full size, the row ring only needs two slots
        PipeLayout pl;
        switch (shape) {
            case kNarrow6:
                if (pipe_layout(p, G, 6, 70 * 1024, pl)) {
                    set_stagger<P, 6, 3>(p);
                    return launch_pipe<QUANT, OUT, P, 6, 1, 4, 3, ADD>(p, pl, stream);
                }
                return kNoFit;
            case kNarrow4:  // two loaders: rows of 3-4 KB without extra rows (fp32 rows at D 768 / 1024)
                if (pipe_layout(p, G, 5, 70 * 1024, pl)) {
                    set_stagger<P, 5, 3>(p);
                    return launch_pipe<QUANT, OUT, P, 5, (G >= 2 ? 2 : 1), 4, 3, ADD>(p, pl, stream);
                }
                return kNoFit;
            case kMid:  // 110 KB x 2 CTAs/SM: two full-size tiles of narrow rows + base row + position row (config 2 "both": 56 us
                        // against 70 us for the single-ring kernel and 75 us for one 200 KB CTA per SM)
                if (pipe_layout(p, G, 4, 110 * 1024, pl)) return launch_pipe<QUANT, OUT, P, 4, (G >= 2 ? 2 : 1), 8, 2, ADD>(p, pl, stream);
                return kNoFit;
            case kWide:
            case kWide3:
            case kWide2:
                if (pipe_layout(p, G, 6, 200 * 1024, pl)) return launch_pipe<QUANT, OUT, P, 6, (G >= 4 ? 4 : G), 12, 1, ADD>(p, pl, stream);
                return kNoFit;
            case kSmall:
                if (pipe_layout(p, G, 2, 70 * 1024, pl)) return launch_pipe<QUANT, OUT, P, 2, 1, 6, 3, ADD>(p, pl, stream);
                return kNoFit;
            default:
                return launch_ldg<QUANT, OUT, P, 4, 2, 6, 4>(p, stream);
        }
    }
    switch (shape) {
        case kNarrow6:
            if (bulk_layout(p, G, 6, 70 * 1024, lay)) {
                set_stagger<P, 6, 3>(p);
                return launch_bulk<QUANT, OUT, P, 6, 4, 3, ADD>(p, lay, stream);
            }
            return kNoFit;
        case kNarrow4:
            if (bulk_layout(p, G, 4, 70 * 1024, lay)) {
                set_stagger<P, 4, 3>(p);
                return launch_bulk<QUANT, OUT, P, 4, 4, 3, ADD>(p, lay, stream);
            }
            return kNoFit;
        case kWide:
            if (bulk_layout(p, G, 6, 200 * 1024, lay)) return launch_bulk<QUANT, OUT, P, 6, 12, 1, ADD>(p, lay, stream);
            return kNoFit;
        case kWide3:
            if (bulk_layout(p, G, 3, 200 * 1024, lay)) return launch_bulk<QUANT, OUT, P, 3, 12, 1, ADD>(p, lay, stream);
            return kNoFit;
        case kWide2:
            if (bulk_layout(p, G, 2, 200 * 1024, lay)) return launch_bulk<QUANT, OUT, P, 2, 12, 1, ADD>(p, lay, stream);
            return kNoFit;
        case kMid:
            if (bulk_layout(p, G, 4, 100 * 1024, lay)) return launch_bulk<QUANT, OUT, P, 4, 8, 2, ADD>(p, lay, stream);
            return kNoFit;
        case kSmall:
            if (bulk_layout(p, G, 2, 70 * 1024, lay)) return launch_bulk<QUANT, OUT, P, 2, 6, 3, ADD>(p, lay, stream);
            return kNoFit;
        default:
            return launch_ldg<QUANT, OUT, P, 4, 2, 6, 4>(p, stream);
    }
}

template <int QUANT, int OUT>
static int launch_p(int P, EmbedParams &p, cudaStream_t stream, int shape) {
    if (p.additive) {  // additive kernels exist for 4 and 8 lanes per position only (any P >= the vocabulary's is valid)
        if (P <= 4) return launch<QUANT, OUT, 4, true>(p, stream, shape);
        return launch<QUANT, OUT, 8, true>(p, stream, shape);
    }
    switch (P) {
        case 1: return launch<QUANT, OUT, 1, false>(p, stream, shape);
        case 2: return launch<QUANT, OUT, 2, false>(p, stream, shape);
        case 4: return launch<QUANT, OUT, 4, false>(p, stream, shape);
        default: return launch<QUANT, OUT, 8, false>(p, stream, shape);
    }
}

}  // namespace scone
