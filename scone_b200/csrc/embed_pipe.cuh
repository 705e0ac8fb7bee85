// embed_pipe.cuh -- the fused path as a THREE-role pipeline (included by embed_kernels.cuh).
//
//   matcher warps  --(fid, token, len) per position-->  metadata ring  --> loader warp --TMA bulk copies--> row ring --> gather warps
//
// embed_bulk_kernel lets the matcher that resolved a tile also stage its rows, so the row ring must hold at least one tile
// per matcher and a matcher can run no further ahead than the ring is deep.  With extra rows per position (fused position
// add: +2 D bytes, additive combine: +2 D bytes) a tile of 8 positions no longer fitted, tiles shrank to 4 positions, and
// the kernel became matcher-bound: the dependent chain ids -> hash -> slot (-> re-probe) costs the same ~6 us for a tile of
// 4 as for a tile of 8 (config 2 + wpe: 12 matchers x 4 positions per chain = 8 positions / us / SM for 442 positions per
// SM = ~52 us, which is what it measured).
// Here the two rings are separate:
//   * matchers only resolve: they write 9 bytes per position into a metadata ring of 4 x NM tiles and never wait for row
//     storage, so tiles stay at the full G = 32 / P positions whatever a position's rows weigh, and the probe chains of
//     many tiles are in flight;
//   * NL loader warps walk the CTA's tiles in order, wait for a free row slot and issue the bulk copies (position g of a tile
//     is staged by loader g % NL: table or fallback row [+ base row of a hit]).  Every loader takes part in
//     every tile, so the row ring only needs two slots and no slot-ownership rule.  Why several: a cp.async.bulk costs
//     ~80 ns to issue and the issues of one warp serialise -- with three rows per position ONE loader spent 1.9 us per
//     tile of 8 positions and capped config 2 + base row + wpe at 104 us (profiles/tune_r02.md).  For the same reason the
//     position rows of a tile are ONE copy: its G positions are consecutive in their sequence, so their wpe rows are one
//     contiguous block of G x 2 D bytes (two blocks where the tile straddles the end of a sequence);
//   * gather warps are those of embed_bulk_kernel; the one that owns a tile's first position also writes the tile's
//     fgram_id / match_len (from the slot header), so matchers and loader never write global memory: with
//     SCONE_EMBED_INPUTS_STABLE they run under the previous kernel's tail without ever waiting for it.
#pragma once

namespace scone {

// ADD (compile time) = the additive combine: measured as a run-time flag it cost the plain path 1-7 % (config 1 6.56 vs
// 6.28 us, config 2 + wpe 57.2 vs 53.1 us, config 3 1017 vs 1006 us), so the plain kernels do not carry it.
template <int QUANT, int OUT, int P, int NM, int NL, int NG, int MINB, bool ADD>
__global__ void __launch_bounds__(32 * (NM + NL + NG), MINB) embed_pipe_kernel(const EmbedParams p, const PipeLayout lay) {
    constexpr int G = 32 / P;
    const int add_off = ADD ? lay.add_off : 0;
    extern __shared__ __align__(128) uint8_t smem[];
    uint64_t *full_bar = reinterpret_cast<uint64_t *>(smem);
    uint64_t *empty_bar = full_bar + kMaxRing;
    uint64_t *meta_full = empty_bar + kMaxRing;
    uint64_t *meta_empty = meta_full + kMaxMetaRing;
    int2 *hdr = reinterpret_cast<int2 *>(meta_empty + kMaxMetaRing);  // [ring][G]   (row id or < 0, fallback / base token or -1)
    int2 *meta = hdr + kMaxRing * G;                                  // [meta_ring][G]
    uint8_t *hdr_len = reinterpret_cast<uint8_t *>(meta + kMaxMetaRing * G);
    uint8_t *meta_len = hdr_len + kMaxRing * G;
    uint8_t *rows_smem = smem + pipe_header_bytes(G);
    const int R = lay.ring, MR = lay.meta_ring;

    asm volatile("griddepcontrol.launch_dependents;");
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) {
        for (int q = 0; q < R; ++q) {
            mbar_init(&full_bar[q], NL);  // one arrival (+ its bytes) per loader
            mbar_init(&empty_bar[q], NG);
        }
        for (int q = 0; q < MR; ++q) {
            mbar_init(&meta_full[q], 1);
            mbar_init(&meta_empty[q], NL);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    // see embed_bulk_kernel: without the flag nothing may run before the previous grid has completed; with it only the
    // gather warps (the only writers of global memory here) wait, just before their first store
    const bool early = (p.flags & SCONE_EMBED_INPUTS_STABLE) != 0;
    if (!early) griddep_wait();

    if (warp < NM) {
        // ===== matcher warps: resolve every NM-th tile of the CTA, publish 9 bytes per position =====
        const int back = p.ix.max_n - 1;
        int64_t it = warp;
        int64_t tile = blockIdx.x + it * gridDim.x;
        int32_t wtok = -1;
        if (!p.fgram_in && tile < p.num_tiles) wtok = load_window_token<P>(p.ids, p.T, tile * G, lane, back);
        if (!p.fgram_in) {
            const unsigned wait_ns = (unsigned)(warp * p.stagger_ns);
            if (wait_ns) __nanosleep(wait_ns);
        }
        for (; tile < p.num_tiles; it += NM, tile += (int64_t)NM * gridDim.x) {
            const int ms = (int)(it % MR);
            const Resolved r = resolve_position<P>(p, ADD, tile, tile + (int64_t)NM * gridDim.x, lane, back, wtok);
            mbar_wait(&meta_empty[ms], (uint32_t)(((it / MR) & 1) ^ 1));
            // lane 0 publishes the whole tile and then arrives: one producer thread per phase
#pragma unroll
            for (int g = 0; g < G; ++g) {
                const int32_t f = __shfl_sync(0xFFFFFFFFu, r.fid, g * P);
                const int32_t k2 = __shfl_sync(0xFFFFFFFFu, r.tok, g * P);
                const int32_t l2 = __shfl_sync(0xFFFFFFFFu, r.len, g * P);
                if (lane == 0) {
                    meta[ms * G + g] = make_int2(f, k2);
                    meta_len[ms * G + g] = (uint8_t)l2;
                }
            }
            if (lane == 0) mbar_arrive(&meta_full[ms]);
        }
    } else if (warp < NM + NL) {
        // ===== loader warps: tiles in order; lane g of loader g % NL stages position g of the tile =====
        const int ld = warp - NM;
        const uint64_t pol = policy_evict_first(), pol_keep = policy_evict_last();
        int64_t itl = 0;
        for (int64_t tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++itl) {
            const int ms = (int)(itl % MR), q = (int)(itl % R);
            mbar_wait(&meta_full[ms], (uint32_t)((itl / MR) & 1));
            int2 e = make_int2(-1, -1);
            int32_t len = 0;
            if (lane < G) {
                e = meta[ms * G + lane];
                len = meta_len[ms * G + lane];
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&meta_empty[ms]);  // the entries are in registers: the matcher may reuse the slot
            const int64_t i = tile * G + lane;
            const bool owner = lane < G && (lane % NL) == ld && i < p.T;
            const uint8_t *src = nullptr, *src3 = nullptr;
            uint32_t bytes = 0;
            if (owner) {
                if (e.x >= 0) {
                    src = row_ptr(p, e.x);
                    bytes = (uint32_t)p.row_stride;
                    if (add_off && e.y >= 0) src3 = p.base + (int64_t)e.y * p.D * 2;  // additive combine: the hit's base row rides along
                } else if (e.y >= 0) {
                    src = p.base + (int64_t)e.y * p.D * 2;
                    bytes = (uint32_t)p.D * 2u;
                }
            }
            // fused position add: the tile's position rows, staged as one block by an otherwise idle lane of the last loader
            const int64_t i0 = tile * G;
            const int npos = (lay.pos_off && ld == NL - 1 && lane == 31) ? (int)(p.T - i0 < G ? p.T - i0 : G) : 0;
            uint32_t total = bytes + (src3 ? (uint32_t)p.D * 2u : 0u) + (uint32_t)npos * (uint32_t)p.D * 2u;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) total += __shfl_xor_sync(0xFFFFFFFFu, total, o);
            mbar_wait(&empty_bar[q], (uint32_t)(((itl / R) & 1) ^ 1));
            if (ld == 0) {  // the slot header is written by one thread, before its arrival
#pragma unroll
                for (int g = 0; g < G; ++g) {
                    const int32_t f = __shfl_sync(0xFFFFFFFFu, e.x, g);
                    const int32_t k2 = __shfl_sync(0xFFFFFFFFu, e.y, g);
                    const int32_t l2 = __shfl_sync(0xFFFFFFFFu, len, g);
                    if (lane == 0) {
                        hdr[q * G + g] = make_int2(f, k2);
                        hdr_len[q * G + g] = (uint8_t)l2;
                    }
                }
            }
            if (lane == 0) mbar_arrive_expect_tx(&full_bar[q], total);
            __syncwarp();
            uint8_t *tile_smem = rows_smem + (size_t)q * lay.tile_bytes;
            uint8_t *slot = tile_smem + (size_t)lane * lay.slot_bytes;
            if (bytes) bulk_g2s(slot, src, bytes, &full_bar[q], pol);
            if (src3) bulk_g2s(slot + add_off, src3, (uint32_t)p.D * 2u, &full_bar[q], pol);
            if (npos) {
                int64_t cur = pos_in_row(i0, p.L, p.T);
                for (int j = 0; j < npos;) {  // one pass unless the tile crosses the end of a sequence
                    const int seg = (int)(p.L - cur < npos - j ? p.L - cur : npos - j);
                    bulk_g2s(tile_smem + lay.pos_off + (size_t)j * p.D * 2, p.pos + cur * p.D * 2, (uint32_t)seg * (uint32_t)p.D * 2u, &full_bar[q],
                             pol_keep);
                    j += seg;
                    cur = 0;
                }
            }
        }
    } else {
        // ===== gather warps: every warp waits for and releases every tile, in order =====
        bool flagged = false, waited = !early;
        const uint64_t pol = policy_evict_first();
        const int w = warp - NM - NL;
        int64_t itl = 0;
        for (int64_t tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++itl) {
            const int q = (int)(itl % R);
            mbar_wait(&full_bar[q], (uint32_t)((itl / R) & 1));
            if (!waited) {  // rows are staged; the stores below are the first thing that must follow the previous grid
                griddep_wait();
                waited = true;
            }
            const int first = (int)(((int64_t)w - (itl * G) % NG + NG) % NG);
            if (first == 0 && !p.fgram_in && lane < G && tile * G + lane < p.T) {  // the match result of the whole tile, coalesced
                if (p.out_id) p.out_id[tile * G + lane] = hdr[q * G + lane].x;
                if (p.out_len) p.out_len[tile * G + lane] = hdr_len[q * G + lane];
            }
            for (int j = first; j < G; j += NG) {
                const int2 e = hdr[q * G + j];
                const int64_t t = tile * G + j;
                if (t < p.T) {
                    const uint8_t *tile_smem = rows_smem + (size_t)q * lay.tile_bytes;
                    const uint8_t *slot = tile_smem + (size_t)j * lay.slot_bytes;
                    const uint8_t *arow = (add_off && e.x >= 0 && e.y >= 0) ? slot + add_off : nullptr;
                    stream_from_smem<QUANT, OUT>(p, slot, arow, lay.pos_off ? tile_smem + lay.pos_off + (size_t)j * p.D * 2 : nullptr, e.x, e.y,
                                                 p.out + t * p.D * 2, lane, pol);
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
