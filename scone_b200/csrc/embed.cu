// embed.cu -- dispatch and C ABI of the fused hot path (kernels: embed_kernels.cuh, instantiated by embed_inst.cu).
//
// Takes over, per position, get_token_f_grams + f_gram_to_id + get_embeddings + the engine's assemble loop + the wte
// fallback of the reference (scone/tokenization/n_gram_extractor.py:106-126, scone/inference/embedding_cache.py:149-181,
// scone/inference/engine.py:235-266, scone/models/language_model.py:239-243), with Algorithm-2 semantics.
#include <cstdlib>

#include "embed_kernels.cuh"

namespace scone {

// one translation unit per (table format, output type): embed_inst.cu
int embed_launch_q0_0(int P, EmbedParams &p, cudaStream_t stream, int shape);  // FP16 -> bf16
int embed_launch_q1_0(int P, EmbedParams &p, cudaStream_t stream, int shape);  // INT8 -> bf16
int embed_launch_q2_0(int P, EmbedParams &p, cudaStream_t stream, int shape);  // INT4 -> bf16
int embed_launch_q0_1(int P, EmbedParams &p, cudaStream_t stream, int shape);  // FP16 -> fp16
int embed_launch_q1_1(int P, EmbedParams &p, cudaStream_t stream, int shape);  // INT8 -> fp16
int embed_launch_q2_1(int P, EmbedParams &p, cudaStream_t stream, int shape);  // INT4 -> fp16
int embed_launch_q3_0(int P, EmbedParams &p, cudaStream_t stream, int shape);  // FP32 -> bf16
int embed_launch_q3_1(int P, EmbedParams &p, cudaStream_t stream, int shape);  // FP32 -> fp16
static_assert(SCONE_QUANT_FP16 == 0 && SCONE_QUANT_INT8 == 1 && SCONE_QUANT_INT4 == 2 && SCONE_QUANT_FP32 == 3 && SCONE_OUT_BF16 == 0 &&
                  SCONE_OUT_FP16 == 1,
              "the embed_launch_q<quant>_<out> names encode these values");

static int dispatch_one(int P, EmbedParams &p, int quant, int out_dtype, cudaStream_t stream, int shape) {
    if (out_dtype == SCONE_OUT_BF16) {
        if (quant == SCONE_QUANT_FP16) return embed_launch_q0_0(P, p, stream, shape);
        if (quant == SCONE_QUANT_INT8) return embed_launch_q1_0(P, p, stream, shape);
        if (quant == SCONE_QUANT_INT4) return embed_launch_q2_0(P, p, stream, shape);
        return embed_launch_q3_0(P, p, stream, shape);
    }
    if (quant == SCONE_QUANT_FP16) return embed_launch_q0_1(P, p, stream, shape);
    if (quant == SCONE_QUANT_INT8) return embed_launch_q1_1(P, p, stream, shape);
    if (quant == SCONE_QUANT_INT4) return embed_launch_q2_1(P, p, stream, shape);
    return embed_launch_q3_1(P, p, stream, shape);
}

// P = the fewest lanes per position the vocabulary needs.
static int dispatch(int P, EmbedParams &p, int quant, int out_dtype, cudaStream_t stream) {
    const int64_t moved = 2ll * p.D + p.row_stride;  // bytes moved per position: the stored row (or a 2 D fallback row) in, 2 D out
    const int narrow[] = {kNarrow6, kNarrow4, kMid, kSmall}, wide[] = {kWide, kWide3, kWide2, kSmall};
    const int *order = moved >= 6144 ? wide : narrow;
    const int n_order = 4;
    int rc = kNoFit;
    if (p.additive && P < 4) P = 4;  // see launch_p
    // Two kernels (measured, profiles/tune_r02.md): the plain path runs fastest on embed_bulk_kernel (one ring, the matcher
    // stages its own tile: fewest hand-offs); with extra rows per position (fused position add, additive combine) the
    // three-role pipeline of embed_pipe.cuh keeps full-size tiles and wins.  SCONE_EMBED_PIPE=0 / 1 forces one of them
    // (read per call so that the tests can run both everywhere).
    // Measured (config 2 / config 3, us per step, bulk vs pipeline): plain 38.4 / 41.5 and 1004 / 1067; + wpe 51.9 / 47.0 and
    // 1530 / 1515; + base row 54.2 / 51.4 and 1625 / 1554; both 70.3 / 56.3 and 2383 / 2295.
    // Plain path with fp32 rows of 2-6 KB (the reference's own row format at D 768 .. 1536): a position moves twice as many
    // bytes in as out, the single ring holds two tiles or fewer for its matchers, and the pipeline wins as well (us per step at
    // D 768 / 1024 / 1280 / 1536: 52.9 -> 48.2, 66.4 -> 61.1, 92.2 -> 76.8, 102.2 -> 90.9; FP16 / INT8 / INT4 rows of any width
    // and fp32 rows of 8 KB stay 1-4 % faster on the single ring: profiles/tune_r02.md section 17).
    const char *pe = getenv("SCONE_EMBED_PIPE");
    const bool extra_rows = p.pos != nullptr || p.additive != 0;
    const bool heavy_rows = p.row_stride > 2ll * p.D && p.row_stride > 2048 && p.row_stride <= 6144;
    if (pe ? pe[0] != '0' : (extra_rows || heavy_rows)) p.flags |= kEmbedPipe;
    if (p.flags & kEmbedPipe) {
        // full-size tiles on any shape before smaller tiles: the pipeline's matchers do not depend on the row ring
        const int plain[] = {kNarrow4, kNarrow6, kMid, kWide, kSmall}, pn[] = {kNarrow6, kMid, kWide, kSmall}, pw[] = {kMid, kWide, kSmall};
        const int *po = !extra_rows ? plain : moved >= 6144 ? pw : pn;
        const int n_po = !extra_rows ? 5 : moved >= 6144 ? 3 : 4;
        for (int pp = P; pp <= 8 && rc == kNoFit; pp <<= 1)
            for (int s = 0; s < n_po && rc == kNoFit; ++s) rc = dispatch_one(pp, p, quant, out_dtype, stream, po[s]);
    }
    for (int s = 0; s < n_order && rc == kNoFit; ++s)
        for (int pp = P; pp <= 8 && rc == kNoFit; pp <<= 1) {
            rc = dispatch_one(pp, p, quant, out_dtype, stream, order[s]);
            if (order[s] == kNarrow6) break;  // only worth it at full tile size
        }
    if (rc == kNoFit) rc = dispatch_one(P, p, quant, out_dtype, stream, kLdg);
    if (rc != SCONE_OK) return rc;
    SCONE_LAUNCHED();
    return SCONE_OK;
}

int check_table(const scone_table_desc_t *t, const char *who);  // table.cu

static int fill_table(EmbedParams &p, const scone_table_desc_t *t, const char *who) {
    int rc = check_table(t, who);
    if (rc != SCONE_OK) return rc;
    p.rows = static_cast<const uint8_t *>(t->d_rows);
    p.shard_rows = nullptr;
    p.world = 1;
    p.row_stride = t->row_stride;
    p.num_rows = t->num_rows;
    p.D = t->dim;
    p.scale_off = t->scale_offset;
    p.group_shift = 0;
    if (t->quant == SCONE_QUANT_INT4) {
        int g8 = t->group / 8, sh = 0;
        while ((1 << sh) < g8) ++sh;
        p.group_shift = sh;
    }
    return SCONE_OK;
}

}  // namespace scone

using namespace scone;

extern "C" {

static int embed_forward_impl(const scone_index_t *index, const scone_table_desc_t *table, const void *d_base_emb, int64_t base_rows,
                              const void *d_pos_emb, const int64_t *d_ids, int64_t B, int64_t L, void *d_out, int32_t out_dtype,
                              int32_t *d_out_id, uint8_t *d_out_len, uint32_t *d_status, void *stream_, uint32_t flags) {
    cudaStream_t stream = (cudaStream_t)stream_;
    SCONE_REQUIRE(index && table, "scone_embed_forward: NULL index or table");
    SCONE_REQUIRE(out_dtype == SCONE_OUT_BF16 || out_dtype == SCONE_OUT_FP16, "scone_embed_forward: out_dtype must be bf16 or fp16");
    SCONE_REQUIRE(B >= 0 && L >= 0, "scone_embed_forward: negative shape");
    const int64_t T = B * L;
    if (T == 0) return SCONE_OK;
    SCONE_REQUIRE(T < (1ll << 40), "scone_embed_forward: batch too large");
    SCONE_REQUIRE(d_ids && d_out, "scone_embed_forward: NULL ids or out");
    SCONE_REQUIRE(d_base_emb && base_rows > 0, "scone_embed_forward: base embedding table required (fallback rows)");
    SCONE_REQUIRE((((uintptr_t)d_base_emb | (uintptr_t)d_out | (uintptr_t)d_pos_emb) & 15) == 0,
                  "scone_embed_forward: base_emb, pos_emb and out must be 16-byte aligned");
    const scone_index_impl *ix = reinterpret_cast<const scone_index_impl *>(index);
    SCONE_REQUIRE(ix->n <= table->num_rows, "scone_embed_forward: index has %lld f-grams but the table only %lld rows",
                  (long long)ix->n, (long long)table->num_rows);
    EmbedParams p{};
    int rc = fill_table(p, table, "scone_embed_forward");
    if (rc != SCONE_OK) return rc;
    p.ix = view_of(ix, T);
    p.fgram_in = nullptr;
    p.base = static_cast<const uint8_t *>(d_base_emb);
    p.V = base_rows;
    p.pos = static_cast<const uint8_t *>(d_pos_emb);
    p.ids = d_ids;
    p.T = T;
    p.L = L;
    p.out = static_cast<uint8_t *>(d_out);
    p.out_id = d_out_id;
    p.out_len = d_out_len;
    p.status = d_status;
    p.additive = (flags & SCONE_EMBED_ADDITIVE) ? 1 : 0;
    p.flags = flags;
    return dispatch(lanes_per_position(ix->len_mask, ix->max_n), p, table->quant, out_dtype, stream);
}

int scone_embed_forward(const scone_index_t *index, const scone_table_desc_t *table, const void *d_base_emb, int64_t base_rows,
                        const void *d_pos_emb, const int64_t *d_ids, int64_t B, int64_t L, void *d_out, int32_t out_dtype,
                        int32_t *d_out_id, uint8_t *d_out_len, uint32_t *d_status, void *stream) {
    return embed_forward_impl(index, table, d_base_emb, base_rows, d_pos_emb, d_ids, B, L, d_out, out_dtype, d_out_id, d_out_len, d_status,
                              stream, 0);
}

int scone_embed_forward_additive(const scone_index_t *index, const scone_table_desc_t *table, const void *d_base_emb, int64_t base_rows,
                                 const void *d_pos_emb, const int64_t *d_ids, int64_t B, int64_t L, void *d_out, int32_t out_dtype,
                                 int32_t *d_out_id, uint8_t *d_out_len, uint32_t *d_status, void *stream) {
    return embed_forward_impl(index, table, d_base_emb, base_rows, d_pos_emb, d_ids, B, L, d_out, out_dtype, d_out_id, d_out_len, d_status,
                              stream, SCONE_EMBED_ADDITIVE);
}

int scone_embed_forward_ex(const scone_index_t *index, const scone_table_desc_t *table, const void *d_base_emb, int64_t base_rows,
                           const void *d_pos_emb, const int64_t *d_ids, int64_t B, int64_t L, void *d_out, int32_t out_dtype,
                           int32_t *d_out_id, uint8_t *d_out_len, uint32_t *d_status, const scone_embed_opts_t *opts, void *stream) {
    const uint32_t flags = opts ? opts->flags : 0u;
    SCONE_REQUIRE((flags & ~(SCONE_EMBED_ADDITIVE | SCONE_EMBED_INPUTS_STABLE)) == 0, "scone_embed_forward_ex: unknown flag bits 0x%x", flags);
    return embed_forward_impl(index, table, d_base_emb, base_rows, d_pos_emb, d_ids, B, L, d_out, out_dtype, d_out_id, d_out_len, d_status,
                              stream, flags);
}

int scone_embed_forward_sharded(const scone_index_t *index, const scone_table_desc_t *shard, const void *const *d_shard_rows,
                                int32_t world, int64_t total_rows, const void *d_base_emb, int64_t base_rows, const void *d_pos_emb,
                                const int64_t *d_ids, int64_t B, int64_t L, void *d_out, int32_t out_dtype, int32_t *d_out_id,
                                uint8_t *d_out_len, uint32_t *d_status, void *stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    SCONE_REQUIRE(index && shard && d_shard_rows, "scone_embed_forward_sharded: NULL index, shard descriptor or pointer table");
    SCONE_REQUIRE(world >= 1 && world <= 64, "scone_embed_forward_sharded: world %d outside [1, 64]", world);
    SCONE_REQUIRE(out_dtype == SCONE_OUT_BF16 || out_dtype == SCONE_OUT_FP16, "scone_embed_forward_sharded: out_dtype must be bf16 or fp16");
    SCONE_REQUIRE(B >= 0 && L >= 0, "scone_embed_forward_sharded: negative shape");
    const int64_t T = B * L;
    if (T == 0) return SCONE_OK;
    SCONE_REQUIRE(T < (1ll << 40), "scone_embed_forward_sharded: batch too large");
    SCONE_REQUIRE(d_ids && d_out, "scone_embed_forward_sharded: NULL ids or out");
    SCONE_REQUIRE(d_base_emb && base_rows > 0, "scone_embed_forward_sharded: base embedding table required (fallback rows)");
    SCONE_REQUIRE((((uintptr_t)d_base_emb | (uintptr_t)d_out | (uintptr_t)d_pos_emb) & 15) == 0,
                  "scone_embed_forward_sharded: base_emb, pos_emb and out must be 16-byte aligned");
    const scone_index_impl *ix = reinterpret_cast<const scone_index_impl *>(index);
    SCONE_REQUIRE(ix->n <= total_rows, "scone_embed_forward_sharded: index has %lld f-grams but the shards only %lld rows", (long long)ix->n,
                  (long long)total_rows);
    SCONE_REQUIRE((total_rows + world - 1) / world <= shard->num_rows, "scone_embed_forward_sharded: %lld rows over %d shards exceed the shard capacity %lld",
                  (long long)total_rows, world, (long long)shard->num_rows);
    EmbedParams p{};
    scone_table_desc_t geom = *shard;
    if (!geom.d_rows) geom.d_rows = reinterpret_cast<const void *>(uintptr_t(16));  // geometry only; never dereferenced when world > 1
    int rc = fill_table(p, &geom, "scone_embed_forward_sharded");
    if (rc != SCONE_OK) return rc;
    p.shard_rows = reinterpret_cast<const uint8_t *const *>(d_shard_rows);
    p.rows = nullptr;
    p.num_rows = total_rows;
    p.ix = view_of(ix, T);
    p.fgram_in = nullptr;
    p.base = static_cast<const uint8_t *>(d_base_emb);
    p.V = base_rows;
    p.pos = static_cast<const uint8_t *>(d_pos_emb);
    p.ids = d_ids;
    p.T = T;
    p.L = L;
    p.out = static_cast<uint8_t *>(d_out);
    p.out_id = d_out_id;
    p.out_len = d_out_len;
    p.status = d_status;
    p.world = -world;  // negative: always go through the pointer table, even for one shard
    return dispatch(lanes_per_position(ix->len_mask, ix->max_n), p, shard->quant, out_dtype, stream);
}

int scone_embed_gather(const scone_table_desc_t *table, const void *d_base_emb, int64_t base_rows, const void *d_pos_emb,
                       int64_t L, const int64_t *d_ids, const int32_t *d_fgram_id, int64_t T, void *d_out, int32_t out_dtype,
                       uint32_t *d_status, void *stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    SCONE_REQUIRE(table, "scone_embed_gather: NULL table");
    SCONE_REQUIRE(out_dtype == SCONE_OUT_BF16 || out_dtype == SCONE_OUT_FP16, "scone_embed_gather: out_dtype must be bf16 or fp16");
    SCONE_REQUIRE(T >= 0, "scone_embed_gather: negative T");
    if (T == 0) return SCONE_OK;
    SCONE_REQUIRE(d_ids && d_out && d_fgram_id, "scone_embed_gather: NULL buffer");
    SCONE_REQUIRE(d_base_emb && base_rows > 0, "scone_embed_gather: base embedding table required (fallback rows)");
    SCONE_REQUIRE(!d_pos_emb || L > 0, "scone_embed_gather: L required with pos_emb");
    SCONE_REQUIRE((((uintptr_t)d_base_emb | (uintptr_t)d_out | (uintptr_t)d_pos_emb) & 15) == 0,
                  "scone_embed_gather: base_emb, pos_emb and out must be 16-byte aligned");
    EmbedParams p{};
    int rc = fill_table(p, table, "scone_embed_gather");
    if (rc != SCONE_OK) return rc;
    p.fgram_in = d_fgram_id;
    p.base = static_cast<const uint8_t *>(d_base_emb);
    p.V = base_rows;
    p.pos = static_cast<const uint8_t *>(d_pos_emb);
    p.ids = d_ids;
    p.T = T;
    p.L = L > 0 ? L : T;
    p.out = static_cast<uint8_t *>(d_out);
    p.status = d_status;
    return dispatch(4, p, table->quant, out_dtype, stream);
}

}  // extern "C"
