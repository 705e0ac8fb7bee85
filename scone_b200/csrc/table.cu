// table.cu -- the cache table: row geometry, quantise-and-store, dequantising gather.
//
// Takes over EmbeddingCache's storage (scone/inference/embedding_cache.py:49-50, :76-111) and its
// get_embeddings gather (:113-147).  The reference keeps fp32 rows; the three stored formats and
// their formulas are defined in oracle/py_oracle.py (SURVEY.md section 8c) and implemented here
// with the same fp32 operations in the same order, so the stored bits are identical.
#include "index_format.cuh"
#include "row_format.cuh"

namespace scone {

int check_table(const scone_table_desc_t *t, const char *who) {
    SCONE_REQUIRE(t->d_rows != nullptr || t->num_rows == 0, "%s: table rows pointer is NULL", who);
    SCONE_REQUIRE(t->quant >= SCONE_QUANT_FP16 && t->quant <= SCONE_QUANT_FP32, "%s: unknown quant %d", who, t->quant);
    SCONE_REQUIRE(t->dim > 0 && t->dim % 8 == 0, "%s: dim %d must be a positive multiple of 8", who, t->dim);
    SCONE_REQUIRE(t->dim <= (1 << 20), "%s: dim %d too large", who, t->dim);
    SCONE_REQUIRE(t->row_stride > 0 && t->row_stride % 16 == 0, "%s: row_stride %lld must be a positive multiple of 16", who,
                  (long long)t->row_stride);
    SCONE_REQUIRE(((uintptr_t)t->d_rows & 15) == 0, "%s: table rows pointer must be 16-byte aligned", who);
    if (t->quant == SCONE_QUANT_INT4) {
        SCONE_REQUIRE(valid_int4_group(t->group), "%s: INT4 group %d must be a power of two >= 8", who, t->group);
        SCONE_REQUIRE(t->dim % t->group == 0, "%s: dim %d not a multiple of group %d", who, t->dim, t->group);
    }
    const int64_t payload = payload_bytes(t->quant, t->dim), scales = scale_bytes(t->quant, t->dim, t->group);
    if (scales)  // the scales may sit anywhere past the payload, aligned
        SCONE_REQUIRE(t->scale_offset >= payload && t->scale_offset % scale_align(t->quant) == 0, "%s: %s scale_offset %d invalid", who,
                      t->quant == SCONE_QUANT_INT8 ? "INT8" : "INT4", t->scale_offset);
    const int64_t need = scales ? t->scale_offset + scales : payload;
    SCONE_REQUIRE(t->row_stride >= need, "%s: row_stride %lld smaller than the %lld bytes a row needs", who,
                  (long long)t->row_stride, (long long)need);
    return SCONE_OK;
}

__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xFFFFFFFFu, v, o));
    return v;
}

// One warp per row.  fp32 operations mirror oracle/py_oracle.py: quant_fp16 / quant_int8_row /
// quant_int4_group (IEEE division, rint = round-half-even).
template <int QUANT>
__global__ void __launch_bounds__(256) store_kernel(uint8_t *rows, int64_t row_stride, int64_t num_rows, int D, int group,
                                                    int scale_off, const float *__restrict__ src, const int64_t *__restrict__ row_ids,
                                                    int64_t row_base, int64_t k, uint32_t *bad) {
    const int lane = threadIdx.x & 31;
    const int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (r >= k) return;
    const int64_t dst_row = row_ids ? row_ids[r] : row_base + r;
    if (dst_row < 0 || dst_row >= num_rows) {
        if (lane == 0 && bad) atomicAdd(bad, 1u);
        return;
    }
    const float *x = src + r * D;
    uint8_t *o = rows + dst_row * row_stride;
    if (QUANT == SCONE_QUANT_FP32) {  // unquantised: the reference's own storage (embedding_cache.py:99, :111)
        for (int d = lane * 4; d < D; d += 128) *reinterpret_cast<float4 *>(o + d * 4) = *reinterpret_cast<const float4 *>(x + d);
    } else if (QUANT == SCONE_QUANT_FP16) {
        for (int d = lane * 2; d < D; d += 64) {
            const float2 v = *reinterpret_cast<const float2 *>(x + d);
            *reinterpret_cast<__half2 *>(o + d * 2) = __floats2half2_rn(v.x, v.y);
        }
    } else if (QUANT == SCONE_QUANT_INT8) {
        float amax = 0.0f;
        for (int d = lane; d < D; d += 32) amax = fmaxf(amax, fabsf(x[d]));
        amax = warp_max(amax);
        const float s = int8_row_scale(amax);
        for (int d = lane * 4; d < D; d += 128) {
            const float4 v = *reinterpret_cast<const float4 *>(x + d);
            const float q[4] = {v.x, v.y, v.z, v.w};
            uint32_t packed = 0;
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                float t = rintf(__fdiv_rn(q[e], s));
                t = fminf(fmaxf(t, -127.0f), 127.0f);
                packed |= ((uint32_t)(int)t & 0xFFu) << (8 * e);
            }
            *reinterpret_cast<uint32_t *>(o + d) = packed;
        }
        if (lane == 0) *reinterpret_cast<float *>(o + scale_off) = s;
    } else {
        // a group of `group` elements is handled by the whole warp, group/32 elements per lane
        // (group >= 64) or by a sub-warp; keep it simple and exact: loop groups, lanes stride by 2.
        const int ngroups = D / group;
        for (int g = 0; g < ngroups; ++g) {
            const float *xg = x + g * group;
            float amax = 0.0f;
            for (int d = lane; d < group; d += 32) amax = fmaxf(amax, fabsf(xg[d]));
            amax = warp_max(amax);
            const __half s16 = int4_group_scale(amax);
            const float sw = __half2float(s16);
            for (int d = lane * 2; d < group; d += 64) {
                float a = fminf(fmaxf(rintf(__fdiv_rn(xg[d], sw)), -7.0f), 7.0f);
                float b = fminf(fmaxf(rintf(__fdiv_rn(xg[d + 1], sw)), -7.0f), 7.0f);
                o[(g * group + d) >> 1] = (uint8_t)(((int)a + 8) | (((int)b + 8) << 4));
            }
            if (lane == 0) *reinterpret_cast<__half *>(o + scale_off + 2 * g) = s16;
        }
    }
}

// One warp per requested row: out[r] = dequant(table[ids[r]]) as fp32 / bf16 / fp16.
template <int QUANT, int OUT>
__global__ void __launch_bounds__(256) gather_kernel(const uint8_t *__restrict__ rows, int64_t row_stride, int64_t num_rows, int D,
                                                     int group_shift, int scale_off, const int64_t *__restrict__ ids, int64_t k,
                                                     uint8_t *__restrict__ out, uint32_t *status) {
    const int lane = threadIdx.x & 31;
    const int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (r >= k) return;
    const int64_t id = ids[r];
    const bool ok = id >= 0 && id < num_rows;
    if (!ok && lane == 0 && status) atomicOr(status, SCONE_STATUS_TOKEN_OOR);
    const uint8_t *row = rows + (ok ? id : 0) * row_stride;
    const int nchunks = D >> 3;
    constexpr int OB = sizeof(OutChunk<OUT>) / 8;  // output bytes per element
    const GlobalRows mem;
    for (int c = lane; c < nchunks; c += 32) {
        f32x8 x;
        if (!ok) zero8(x);
        else decode_chunk<QUANT>(load_chunk<QUANT>(mem, row, c, scale_off, group_shift, row_scale<QUANT>(mem, row, scale_off)), x);
        *reinterpret_cast<OutChunk<OUT> *>(out + ((int64_t)r * D + c * 8) * OB) = pack_chunk<OUT>(x);
    }
}

// One warp per requested row: copy row_stride bytes verbatim (16 B vectors, 4 in flight per lane).
__global__ void __launch_bounds__(256) gather_packed_kernel(const uint8_t *__restrict__ rows, int64_t row_stride, int64_t num_rows,
                                                            const int32_t *__restrict__ ids, int64_t k, uint8_t *__restrict__ out,
                                                            uint32_t *status) {
    const int lane = threadIdx.x & 31;
    const int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (r >= k) return;
    const int32_t id = __ldg(ids + r);
    const bool ok = id >= 0 && id < num_rows;
    if (!ok && lane == 0 && status) atomicOr(status, SCONE_STATUS_TOKEN_OOR);
    const uint8_t *src = rows + (int64_t)(ok ? id : 0) * row_stride;
    uint8_t *dst = out + r * row_stride;
    const int nvec = (int)(row_stride >> 4);
    const uint64_t pol = policy_evict_first();
    for (int c0 = lane; c0 < nvec; c0 += 128) {
        uint4 v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int c = c0 + 32 * u;
            v[u] = make_uint4(0u, 0u, 0u, 0u);
            if (c < nvec && ok) v[u] = ldg_stream_16(src + c * 16, pol);
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int c = c0 + 32 * u;
            if (c < nvec) *reinterpret_cast<uint4 *>(dst + c * 16) = v[u];
        }
    }
}

// Reference-code semantics: one warp per position, mean of the rows of every f-gram containing it.
// all_ids[t, n-1] = id of the n-gram ENDING at flat position t (scone_index_match_all).
template <int QUANT, int OUT>
__global__ void __launch_bounds__(256) mean_kernel(const uint8_t *__restrict__ rows, int64_t row_stride, int D, int group_shift,
                                                   int scale_off, const int32_t *__restrict__ all_ids, int max_n, int64_t T, int64_t L,
                                                   uint8_t *__restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t t = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (t >= T) return;
    const int64_t pos = t % L;
    // the containing f-grams, in the reference's list order: n ascending, start ascending
    int32_t ids[28];
    int k = 0;
    for (int n = 1; n <= max_n; ++n) {
        for (int s = n - 1; s >= 0; --s) {  // start = pos - s ascending  <=>  end = pos - s + n - 1 ascending
            const int64_t e = pos - s + n - 1;
            if (pos - s < 0 || e >= L) continue;
            const int32_t id = __ldg(all_ids + (t - s + n - 1) * max_n + (n - 1));
            if (id >= 0) ids[k++] = id;
        }
    }
    const int nchunks = D >> 3;
    constexpr int OB = sizeof(OutChunk<OUT>) / 8;  // output bytes per element
    const GlobalRows mem;
    for (int c = lane; c < nchunks; c += 32) {
        f32x8 acc;
        zero8(acc);
        for (int r = 0; r < k; ++r) {
            const uint8_t *row = rows + (int64_t)ids[r] * row_stride;
            f32x8 x;
            decode_chunk<QUANT>(load_chunk<QUANT>(mem, row, c, scale_off, group_shift, row_scale<QUANT>(mem, row, scale_off)), x);
            add8(acc, x);
        }
        if (k > 1) {
#pragma unroll
            for (int e = 0; e < 4; ++e) acc[e] = make_float2(__fdiv_rn(acc[e].x, (float)k), __fdiv_rn(acc[e].y, (float)k));
        }
        *reinterpret_cast<OutChunk<OUT> *>(out + (t * D + c * 8) * OB) = pack_chunk<OUT>(acc);
    }
}

}  // namespace scone

using namespace scone;

extern "C" {

int scone_table_layout(int32_t quant, int32_t dim, int32_t group, int32_t align, int64_t *row_stride, int32_t *scale_offset) {
    SCONE_REQUIRE(row_stride && scale_offset, "scone_table_layout: NULL output");
    SCONE_REQUIRE(dim > 0 && dim % 8 == 0, "scone_table_layout: dim %d must be a positive multiple of 8", dim);
    if (align <= 0) align = 32;
    SCONE_REQUIRE(align % 16 == 0, "scone_table_layout: align %d must be a multiple of 16", align);
    SCONE_REQUIRE(quant >= SCONE_QUANT_FP16 && quant <= SCONE_QUANT_FP32, "scone_table_layout: unknown quant %d", quant);
    if (quant == SCONE_QUANT_INT4)
        SCONE_REQUIRE(valid_int4_group(group) && dim % group == 0,
                      "scone_table_layout: INT4 needs a power-of-two group >= 8 dividing dim (group %d, dim %d)", group, dim);
    const int64_t payload = payload_bytes(quant, dim), scales = scale_bytes(quant, dim, group);
    *row_stride = (payload + scales + align - 1) / align * align;
    *scale_offset = scales ? (int32_t)payload : 0;  // right after the payload, aligned as dim is a multiple of 8
    return SCONE_OK;
}

int scone_table_store(const scone_table_desc_t *table, const float *d_rows_f32, const int64_t *d_row_ids, int64_t row_base,
                      int64_t k, void *stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    SCONE_REQUIRE(table, "scone_table_store: NULL table");
    int rc = check_table(table, "scone_table_store");
    if (rc != SCONE_OK) return rc;
    SCONE_REQUIRE(k >= 0, "scone_table_store: negative k");
    if (k == 0) return SCONE_OK;
    SCONE_REQUIRE(d_rows_f32, "scone_table_store: NULL source rows");
    SCONE_REQUIRE(((uintptr_t)d_rows_f32 & 15) == 0, "scone_table_store: source rows must be 16-byte aligned");
    SCONE_REQUIRE(d_row_ids || (row_base >= 0 && row_base + k <= table->num_rows), "scone_table_store: rows [%lld, %lld) outside the table",
                  (long long)row_base, (long long)(row_base + k));
    uint8_t *rows = static_cast<uint8_t *>(const_cast<void *>(table->d_rows));
    SCONE_GRID(blocks, (k + 7) / 8, "scone_table_store");
    with_constant<SCONE_QUANT_FP16, SCONE_QUANT_INT8, SCONE_QUANT_INT4, SCONE_QUANT_FP32>(table->quant, [&](auto q) {
        store_kernel<q()><<<blocks, 256, 0, stream>>>(rows, table->row_stride, table->num_rows, table->dim, table->group, table->scale_offset,
                                                      d_rows_f32, d_row_ids, row_base, k, nullptr);
    });
    SCONE_LAUNCHED();
    return SCONE_OK;
}

int scone_embed_mean_forward(const scone_index_t *index, const scone_table_desc_t *table, const int64_t *d_ids, int64_t B, int64_t L,
                             int32_t *d_work, void *d_out, int32_t out_dtype, void *stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    SCONE_REQUIRE(index && table, "scone_embed_mean_forward: NULL index or table");
    int rc = check_table(table, "scone_embed_mean_forward");
    if (rc != SCONE_OK) return rc;
    SCONE_REQUIRE(out_dtype >= SCONE_OUT_BF16 && out_dtype <= SCONE_OUT_FP32, "scone_embed_mean_forward: unknown out_dtype %d", out_dtype);
    SCONE_REQUIRE(B >= 0 && L >= 0, "scone_embed_mean_forward: negative shape");
    const int64_t T = B * L;
    if (T == 0) return SCONE_OK;
    SCONE_REQUIRE(d_ids && d_work && d_out, "scone_embed_mean_forward: NULL buffer");
    const scone_index_impl *ix = reinterpret_cast<const scone_index_impl *>(index);
    SCONE_REQUIRE(ix->n <= table->num_rows, "scone_embed_mean_forward: index has more f-grams than the table has rows");
    rc = scone_index_match_all(index, d_ids, B, L, d_work, stream_);
    if (rc != SCONE_OK) return rc;
    SCONE_GRID(blocks, (T + 7) / 8, "scone_embed_mean_forward");
    with_constant<SCONE_QUANT_FP16, SCONE_QUANT_INT8, SCONE_QUANT_INT4, SCONE_QUANT_FP32>(table->quant, [&](auto q) {
        with_constant<SCONE_OUT_BF16, SCONE_OUT_FP16, SCONE_OUT_FP32>(out_dtype, [&](auto o) {
            mean_kernel<q(), o()><<<blocks, 256, 0, stream>>>(static_cast<const uint8_t *>(table->d_rows), table->row_stride, table->dim,
                                                              group_shift(table->group), table->scale_offset, d_work, ix->v.max_n, T, L,
                                                              static_cast<uint8_t *>(d_out));
        });
    });
    SCONE_LAUNCHED();
    return SCONE_OK;
}

int scone_table_gather_packed(const scone_table_desc_t *table, const int32_t *d_row_ids, int64_t k, void *d_out, uint32_t *d_status,
                              void *stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    SCONE_REQUIRE(table, "scone_table_gather_packed: NULL table");
    int rc = check_table(table, "scone_table_gather_packed");
    if (rc != SCONE_OK) return rc;
    SCONE_REQUIRE(k >= 0, "scone_table_gather_packed: negative k");
    if (k == 0) return SCONE_OK;
    SCONE_REQUIRE(d_row_ids && d_out, "scone_table_gather_packed: NULL buffer");
    SCONE_REQUIRE(((uintptr_t)d_out & 15) == 0, "scone_table_gather_packed: out must be 16-byte aligned");
    SCONE_GRID(blocks, (k + 7) / 8, "scone_table_gather_packed");
    gather_packed_kernel<<<blocks, 256, 0, stream>>>(static_cast<const uint8_t *>(table->d_rows), table->row_stride, table->num_rows,
                                                    d_row_ids, k, static_cast<uint8_t *>(d_out), d_status);
    SCONE_LAUNCHED();
    return SCONE_OK;
}

int scone_table_gather(const scone_table_desc_t *table, const int64_t *d_row_ids, int64_t k, void *d_out, int32_t out_dtype,
                       uint32_t *d_status, void *stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    SCONE_REQUIRE(table, "scone_table_gather: NULL table");
    int rc = check_table(table, "scone_table_gather");
    if (rc != SCONE_OK) return rc;
    SCONE_REQUIRE(out_dtype >= SCONE_OUT_BF16 && out_dtype <= SCONE_OUT_FP32, "scone_table_gather: unknown out_dtype %d", out_dtype);
    SCONE_REQUIRE(k >= 0, "scone_table_gather: negative k");
    if (k == 0) return SCONE_OK;
    SCONE_REQUIRE(d_row_ids && d_out, "scone_table_gather: NULL buffer");
    SCONE_GRID(blocks, (k + 7) / 8, "scone_table_gather");
    with_constant<SCONE_QUANT_FP16, SCONE_QUANT_INT8, SCONE_QUANT_INT4, SCONE_QUANT_FP32>(table->quant, [&](auto q) {
        with_constant<SCONE_OUT_BF16, SCONE_OUT_FP16, SCONE_OUT_FP32>(out_dtype, [&](auto o) {
            gather_kernel<q(), o()><<<blocks, 256, 0, stream>>>(static_cast<const uint8_t *>(table->d_rows), table->row_stride, table->num_rows,
                                                                table->dim, group_shift(table->group), table->scale_offset, d_row_ids, k,
                                                                static_cast<uint8_t *>(d_out), d_status);
        });
    });
    SCONE_LAUNCHED();
    return SCONE_OK;
}

}  // extern "C"
