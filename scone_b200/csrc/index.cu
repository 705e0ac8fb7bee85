// index.cu -- the device-resident f-gram index: build, audit, longest-match lookup, match-all.
//
// Takes over the Python set / dict of int tuples of the reference's NGramExtractor
// (scone/tokenization/n_gram_extractor.py:41-44, :96-99, :121-122) and the tuple -> id lookup of
// scone/inference/embedding_cache.py:173.
#include <cstdlib>

#include "match.cuh"

namespace scone {

// audit counters read back once at create time
struct BuildStats {
    unsigned long long bad_len;
    unsigned long long bad_tok;
    unsigned long long dup;
    unsigned int len_mask;
    int max_probe;
    int max_tok;
};

// Key and hash of vocabulary row i; returns its length, 0 for a length outside [1, max_n], -1 for a negative token.
__device__ __forceinline__ int vocab_key(const int32_t *__restrict__ tokens, const uint8_t *__restrict__ lens, int64_t i, int32_t max_n,
                                         int32_t (&key)[7], uint64_t &h) {
    const int len = lens[i];
    if (len < 1 || len > max_n) return 0;
    h = hash_seed();
    bool bad = false;
#pragma unroll
    for (int k = 0; k < 7; ++k) {
        key[k] = -1;
        if (k < len) {
            int32_t t = tokens[i * max_n + (len - 1 - k)];
            bad |= t < 0;
            key[k] = t;
            h = hash_roll(h, (uint32_t)t);
        }
    }
    if (bad) return -1;
    h = hash_finish(h, len);
    return len;
}

// First pass: validate the vocabulary and find the largest token (decides the slot format).
__global__ void __launch_bounds__(256) index_scan_kernel(const int32_t *__restrict__ tokens, const uint8_t *__restrict__ lens, int64_t n,
                                                         int32_t max_n, BuildStats *stats) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int32_t key[7];
    uint64_t h;
    const int len = vocab_key(tokens, lens, i, max_n, key, h);
    if (len <= 0) {
        atomicAdd(len == 0 ? &stats->bad_len : &stats->bad_tok, 1ull);
        return;
    }
    int mx = 0;
#pragma unroll
    for (int k = 0; k < 7; ++k) mx = key[k] > mx ? key[k] : mx;
    atomicMax(&stats->max_tok, mx);
}

// One thread per f-gram: set its filter bits and insert it.
__global__ void __launch_bounds__(256) index_build_kernel(const int32_t *__restrict__ tokens, const uint8_t *__restrict__ lens,
                                                          int64_t n, int32_t max_n, IndexView ix, BuildStats *stats) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int32_t key[7];
    uint64_t h;
    const int len = vocab_key(tokens, lens, i, max_n, key, h);
    if (len <= 0) return;  // counted by the scan
    if (ix.filter) atomicOr(&ix.filter[filter_word(h, ix.filter_mask)], filter_bits(h));
    const int probes = ix.format == kSlotCompact20   ? insert<Compact20Slot>(ix.slots, ix.cap, h, key, (uint32_t)i)
                       : ix.format == kSlotCompact16 ? insert<Compact16Slot>(ix.slots, ix.cap, h, key, (uint32_t)i)
                                                     : insert<WideSlot>(ix.slots, ix.cap, h, key, (uint32_t)i);
    atomicOr(&stats->len_mask, 1u << (len - 1));
    atomicMax(&stats->max_probe, probes);
}

// After the build: every f-gram must find ITSELF.  Two rows with the same key resolve to the
// same (first) slot, so the later row sees a different id -> counted as a duplicate.
__global__ void __launch_bounds__(256) index_audit_kernel(const int32_t *__restrict__ tokens, const uint8_t *__restrict__ lens,
                                                          int64_t n, int32_t max_n, IndexView ix, BuildStats *stats) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int32_t key[7];
    uint64_t h;
    if (vocab_key(tokens, lens, i, max_n, key, h) <= 0) return;
    if (probe_any(ix, h, key) != (int32_t)i) atomicAdd(&stats->dup, 1ull);
}

// ---------------------------------------------------------------------------------------------
// standalone match kernels (the fused path in embed.cu uses the same match_window())
// ---------------------------------------------------------------------------------------------
template <int P>
__global__ void __launch_bounds__(256) lookup_kernel(IndexView ix, const int64_t *__restrict__ ids, int64_t T, int64_t L,
                                                     int32_t *__restrict__ out_id, uint8_t *__restrict__ out_len) {
    constexpr int G = 32 / P;
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t base = warp * G;
    if (base >= T) return;
    const int back = ix.max_n - 1;
    WindowMatch m = match_window<P>(ix, load_window_token<P>(ids, T, base, lane, back), T, L, base, lane, back);
    const int j = lane / P;
    if ((lane % P) == 0 && base + j < T) {
        if (out_id) out_id[base + j] = m.fid;
        if (out_len) out_len[base + j] = (uint8_t)m.len;
    }
}

template <int P>
__global__ void __launch_bounds__(256) match_all_kernel(IndexView ix, const int64_t *__restrict__ ids, int64_t T, int64_t L,
                                                        int32_t *__restrict__ out) {
    constexpr int G = 32 / P;
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t base = warp * G;
    if (base >= T) return;
    const int back = ix.max_n - 1;
    const int j = lane / P, n1 = lane % P;  // dense mapping: candidate n1 is length n1 + 1
    const bool present = n1 < ix.max_n && ((ix.len_mask >> n1) & 1u);
    int32_t fid = candidate_id<P>(ix, load_window_token<P>(ids, T, base, lane, back), T, L, base, lane, present ? n1 + 1 : 0, back);
    if (n1 < ix.max_n && base + j < T) out[(base + j) * ix.max_n + n1] = fid;
}

static int lanes_dense(int max_n) { return max_n <= 1 ? 1 : max_n <= 2 ? 2 : max_n <= 4 ? 4 : 8; }

}  // namespace scone

using namespace scone;

extern "C" {

int scone_index_create(const int32_t *d_tokens, const uint8_t *d_lens, int64_t n, int32_t max_n, double load_factor,
                       void *stream_, scone_index_t **out) {
    cudaStream_t stream = (cudaStream_t)stream_;
    SCONE_REQUIRE(out != nullptr, "scone_index_create: out is NULL");
    *out = nullptr;
    SCONE_REQUIRE(n >= 0 && n < kSlotFormats[kSlotWide].n_limit, "scone_index_create: n = %lld outside [0, 2^31-1)", (long long)n);
    SCONE_REQUIRE(max_n >= 1 && max_n <= SCONE_MAX_N, "scone_index_create: max_n = %d outside [1, %d]", max_n, SCONE_MAX_N);
    SCONE_REQUIRE(n == 0 || (d_tokens && d_lens), "scone_index_create: NULL vocabulary arrays");
    SCONE_REQUIRE(!(load_factor > 0.9), "scone_index_create: load_factor %.3f > 0.9", load_factor);

    scone_index_impl *ix = new (std::nothrow) scone_index_impl();
    if (!ix) {
        set_error("scone_index_create: out of host memory");
        return SCONE_E_NOMEM;
    }
    ix->n = n;
    ix->v.max_n = max_n;
    BuildStats *d_stats = nullptr;
    BuildStats h{};
    const unsigned blocks = (unsigned)((n + 255) / 256);
    int rc = [&]() -> int {
        SCONE_CUDA(cudaMalloc(&d_stats, sizeof(BuildStats)));
        SCONE_CUDA(cudaMemsetAsync(d_stats, 0, sizeof(BuildStats), stream));
        // pass 1: validate, find the largest token -> slot format
        if (n > 0) {
            index_scan_kernel<<<blocks, 256, 0, stream>>>(d_tokens, d_lens, n, max_n, d_stats);
            SCONE_LAUNCHED();
        }
        SCONE_CUDA(cudaMemcpyAsync(&h, d_stats, sizeof h, cudaMemcpyDeviceToHost, stream));
        SCONE_CUDA(cudaStreamSynchronize(stream));
        if (h.bad_len || h.bad_tok) return SCONE_OK;  // reported below
        const IndexPlan pl = plan_index(
            IndexCall{n, max_n, h.max_tok, load_factor, getenv("SCONE_INDEX_FORMAT"), getenv("SCONE_INDEX_FILTER")});
        ix->v.format = pl.format;
        ix->v.cap = pl.cap;
        ix->v.filter_mask = pl.filter_words;
        ix->filter_always = pl.filter_always;
        // device buffer filled with `fill` bytes; the pointer stays NULL when the allocation fails
        auto alloc = [&](auto **p, size_t bytes, int fill, const char *what) -> int {
            cudaError_t e = cudaMalloc(p, bytes);
            if (e != cudaSuccess) {
                set_error("scone_index_create: cudaMalloc of %llu %s bytes failed: %s", (unsigned long long)bytes, what, cudaGetErrorString(e));
                *p = nullptr;
                return e == cudaErrorMemoryAllocation ? SCONE_E_NOMEM : SCONE_E_CUDA;
            }
            SCONE_CUDA(cudaMemsetAsync(*p, fill, bytes, stream));
            return SCONE_OK;
        };
        int rc = alloc(&ix->v.slots, pl.cap * kSlotFormats[pl.format].slot_bytes, 0xFF, "slot");  // all-ones: every slot empty
        if (rc == SCONE_OK && pl.filter_words) rc = alloc(&ix->v.filter, (size_t)pl.filter_words * sizeof(uint32_t), 0, "filter");
        if (rc != SCONE_OK) return rc;
        // pass 2: insert, then every f-gram looks itself up (duplicate audit).  Both read the handle's view (its len_mask is
        // not set yet), with the filter: an f-gram the filter rejected would not find itself.
        if (n > 0) {
            index_build_kernel<<<blocks, 256, 0, stream>>>(d_tokens, d_lens, n, max_n, ix->v, d_stats);
            SCONE_LAUNCHED();
            index_audit_kernel<<<blocks, 256, 0, stream>>>(d_tokens, d_lens, n, max_n, ix->v, d_stats);
            SCONE_LAUNCHED();
        }
        SCONE_CUDA(cudaMemcpyAsync(&h, d_stats, sizeof h, cudaMemcpyDeviceToHost, stream));
        SCONE_CUDA(cudaStreamSynchronize(stream));
        return SCONE_OK;
    }();
    if (d_stats) cudaFree(d_stats);
    if (rc == SCONE_OK && (h.bad_len || h.bad_tok || h.dup)) {
        set_error("scone_index_create: vocabulary rejected: %llu duplicated f-grams, %llu lengths outside [1, %d], %llu rows with negative tokens",
                  h.dup, h.bad_len, max_n, h.bad_tok);
        rc = SCONE_E_VOCAB;
    }
    if (rc != SCONE_OK) {
        if (ix->v.slots) cudaFree(ix->v.slots);
        if (ix->v.filter) cudaFree(ix->v.filter);
        delete ix;
        return rc;
    }
    ix->v.len_mask = h.len_mask;
    ix->max_probe = h.max_probe;
    *out = reinterpret_cast<scone_index_t *>(ix);
    return SCONE_OK;
}

int scone_index_destroy(scone_index_t *index) {
    if (!index) return SCONE_OK;
    scone_index_impl *ix = reinterpret_cast<scone_index_impl *>(index);
    cudaError_t e = cudaFree(ix->v.slots);
    const cudaError_t e2 = cudaFree(ix->v.filter);  // NULL (no filter) frees nothing
    if (e == cudaSuccess) e = e2;
    delete ix;
    if (e != cudaSuccess) {
        set_error("scone_index_destroy: cudaFree failed: %s", cudaGetErrorString(e));
        return SCONE_E_CUDA;
    }
    return SCONE_OK;
}

int scone_index_info(const scone_index_t *index, scone_index_info_t *info) {
    SCONE_REQUIRE(index && info, "scone_index_info: NULL argument");
    const scone_index_impl *ix = reinterpret_cast<const scone_index_impl *>(index);
    info->num_fgrams = ix->n;
    info->capacity = (int64_t)ix->v.cap;
    info->filter_bytes = ix->v.filter ? (int64_t)ix->v.filter_mask * 4 : 0;
    info->slot_bytes = kSlotFormats[ix->v.format].slot_bytes;
    info->bytes = (int64_t)ix->v.cap * info->slot_bytes + info->filter_bytes;
    info->max_n = ix->v.max_n;
    info->len_mask = ix->v.len_mask;
    info->max_probe = ix->max_probe;
    info->slot_format = ix->v.format;
    return SCONE_OK;
}

int scone_index_lookup(const scone_index_t *index, const int64_t *d_ids, int64_t B, int64_t L, int32_t *d_out_id,
                       uint8_t *d_out_len, void *stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    SCONE_REQUIRE(index, "scone_index_lookup: NULL index");
    SCONE_REQUIRE(B >= 0 && L >= 0, "scone_index_lookup: negative shape");
    const int64_t T = B * L;
    if (T == 0) return SCONE_OK;
    SCONE_REQUIRE(d_ids, "scone_index_lookup: NULL ids");
    SCONE_REQUIRE(T < (1ll << 40), "scone_index_lookup: batch too large");
    const scone_index_impl *ix = reinterpret_cast<const scone_index_impl *>(index);
    IndexView v = view_of(ix, T);
    const int P = lanes_per_position(ix->v.len_mask, ix->v.max_n);
    const int64_t windows = (T + (32 / P) - 1) / (32 / P);
    SCONE_GRID(blocks, (windows + 7) / 8, "scone_index_lookup");
    switch (P) {
        case 1: lookup_kernel<1><<<blocks, 256, 0, stream>>>(v, d_ids, T, L, d_out_id, d_out_len); break;
        case 2: lookup_kernel<2><<<blocks, 256, 0, stream>>>(v, d_ids, T, L, d_out_id, d_out_len); break;
        case 4: lookup_kernel<4><<<blocks, 256, 0, stream>>>(v, d_ids, T, L, d_out_id, d_out_len); break;
        default: lookup_kernel<8><<<blocks, 256, 0, stream>>>(v, d_ids, T, L, d_out_id, d_out_len); break;
    }
    SCONE_LAUNCHED();
    return SCONE_OK;
}

int scone_index_match_all(const scone_index_t *index, const int64_t *d_ids, int64_t B, int64_t L, int32_t *d_out,
                          void *stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    SCONE_REQUIRE(index, "scone_index_match_all: NULL index");
    SCONE_REQUIRE(B >= 0 && L >= 0, "scone_index_match_all: negative shape");
    const int64_t T = B * L;
    if (T == 0) return SCONE_OK;
    SCONE_REQUIRE(d_ids && d_out, "scone_index_match_all: NULL buffer");
    const scone_index_impl *ix = reinterpret_cast<const scone_index_impl *>(index);
    IndexView v = view_of(ix, T);
    const int P = lanes_dense(ix->v.max_n);
    const int64_t windows = (T + (32 / P) - 1) / (32 / P);
    SCONE_GRID(blocks, (windows + 7) / 8, "scone_index_match_all");
    switch (P) {
        case 1: match_all_kernel<1><<<blocks, 256, 0, stream>>>(v, d_ids, T, L, d_out); break;
        case 2: match_all_kernel<2><<<blocks, 256, 0, stream>>>(v, d_ids, T, L, d_out); break;
        case 4: match_all_kernel<4><<<blocks, 256, 0, stream>>>(v, d_ids, T, L, d_out); break;
        default: match_all_kernel<8><<<blocks, 256, 0, stream>>>(v, d_ids, T, L, d_out); break;
    }
    SCONE_LAUNCHED();
    return SCONE_OK;
}

}  // extern "C"
