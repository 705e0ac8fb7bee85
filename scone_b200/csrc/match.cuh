// match.cuh -- warp-cooperative f-gram matching shared by the standalone lookup and the fused path.
//
// A warp owns a window of G = 32 / P consecutive positions of the flattened [B * L] batch, where
// P = lanes per position = the power of two >= max_n.  Lane j*P + (n-1) probes the n-gram ENDING
// at position base + j; the P candidates of a position are resolved concurrently and the longest
// hit is picked with one ballot (Algorithm 2: n = max_n .. 1, first hit wins).
#pragma once
#include "common.cuh"

namespace scone {

struct WindowMatch {
    int32_t fid;  // -1 = no f-gram ends here
    int32_t len;  // 0 = none
};

// position of flat index i inside its row of length L
__device__ __forceinline__ int64_t pos_in_row(int64_t i, int64_t L, int64_t T) {
    if (T <= 0xFFFFFFFFll) return (int64_t)((uint32_t)i % (uint32_t)L);
    return i % L;
}

// Lane mapping.  A warp owns a tile of G = 32 / P consecutive positions; the P lanes of a position each take one
// candidate length.  `back` = max_n - 1 = how far a candidate reaches behind its position (G + back <= 32).
//   compact mapping (lookup / fused path): candidate c = lane % P is the c-th length PRESENT in the vocabulary
//     (len_mask), so P = pow2 >= popcount(len_mask): a max_n = 5 vocabulary without unigrams needs 4 lanes, not 8.
//   dense mapping (match_all): candidate c is length c + 1, P = pow2 >= max_n.

// Lanes 0 .. G+back-1 hold the tokens base-back .. base+G-1 (as int32; vocabulary tokens are non-negative int32,
// anything else is mapped to -1 and can only miss).
template <int P>
__device__ __forceinline__ int32_t load_window_token(const int64_t *__restrict__ ids, int64_t T, int64_t base, int lane, int back) {
    constexpr int G = 32 / P;
    const int64_t gi = base - back + lane;
    int64_t t64 = -1;
    if (lane < G + back && gi >= 0 && gi < T) t64 = __ldg(ids + gi);
    return (t64 >= 0 && t64 <= 0x7FFFFFFFll) ? (int32_t)t64 : -1;
}

// token of the lane's own position (lane / P) out of the window registers
template <int P>
__device__ __forceinline__ int32_t own_token(int32_t tok, int lane, int back) {
    return __shfl_sync(0xFFFFFFFFu, tok, lane / P + back);
}

// length of compact candidate c (the c-th set bit of len_mask, ascending), 0 if there is none
__device__ __forceinline__ int candidate_len(uint32_t len_mask, int c) {
    const unsigned pos = __fns(len_mask, 0, c + 1);
    return pos > 31u ? 0 : (int)pos + 1;
}

// id of the n-gram ending at the lane's position, or -1 (n = 0: no candidate).  `tok` from load_window_token.
template <int P>
__device__ __forceinline__ int32_t candidate_id(const IndexView &ix, int32_t tok, int64_t T, int64_t L, int64_t base, int lane, int n,
                                                int back) {
    constexpr unsigned FULL = 0xFFFFFFFFu;
    const int j = lane / P;
    const int64_t i = base + j;
    bool cand = n >= 1 && n <= ix.max_n && i < T;
    if (cand) cand = (int64_t)n <= pos_in_row(i, L, T) + 1;  // the n-gram must not cross the row start
    int32_t key[7];
    uint64_t h = hash_seed();
#pragma unroll
    for (int k = 0; k < 7; ++k) key[k] = -1;
#pragma unroll
    for (int k = 0; k < 7; ++k) {
        if (k <= back) {                                           // warp-uniform
            const int32_t t = __shfl_sync(FULL, tok, j + back - k);  // token at position i - k
            if (k < n) {
                key[k] = t;
                cand = cand && t >= 0;
                h = hash_roll(h, (uint32_t)t);
            }
        }
    }
    if (!cand) return -1;
    return probe_any(ix, hash_finish(h, n), key);
}

// Longest hit of the lane's position (compact mapping); every lane of a P-lane group returns the same value.
template <int P>
__device__ __forceinline__ WindowMatch match_window(const IndexView &ix, int32_t tok, int64_t T, int64_t L, int64_t base, int lane,
                                                    int back) {
    constexpr unsigned FULL = 0xFFFFFFFFu;
    const int32_t cid = candidate_id<P>(ix, tok, T, L, base, lane, candidate_len(ix.len_mask, lane % P), back);
    const unsigned hit = __ballot_sync(FULL, cid >= 0);
    const int j = lane / P;
    const unsigned bits = (hit >> (j * P)) & (P == 32 ? 0xFFFFFFFFu : ((1u << P) - 1u));
    WindowMatch m{-1, 0};
    int src = lane;
    if (bits) {
        const int top = 31 - __clz((int)bits);   // candidates are in ascending length order: the highest hit is the longest
        m.len = candidate_len(ix.len_mask, top);
        src = j * P + top;
    }
    const int32_t f = __shfl_sync(FULL, cid, src);
    if (bits) m.fid = f;
    return m;
}

// lanes per position for the compact mapping
inline int lanes_per_position(uint32_t len_mask, int max_n) {
    int c = __builtin_popcount(len_mask), P = 1;
    while (P < c) P <<= 1;
    while (32 / P + max_n - 1 > 32) P <<= 1;  // the token window of a tile must fit the warp
    return P;
}

}  // namespace scone
