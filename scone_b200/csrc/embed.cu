// embed.cu -- dispatch and C ABI of the fused hot path (kernels: embed_kernels.cuh, instantiated by embed_inst.cu).
//
// Takes over, per position, get_token_f_grams + f_gram_to_id + get_embeddings + the engine's assemble loop + the wte
// fallback of the reference (scone/tokenization/n_gram_extractor.py:106-126, scone/inference/embedding_cache.py:149-181,
// scone/inference/engine.py:235-266, scone/models/language_model.py:239-243), with Algorithm-2 semantics.
#include <cstdlib>

#include "embed_kernels.cuh"

namespace scone {

// one translation unit per (table format, output type): embed_inst.cu
using EmbedLaunch = int (*)(const EmbedPlan &, EmbedParams &, cudaStream_t);
int embed_launch_q0_0(const EmbedPlan &, EmbedParams &, cudaStream_t), embed_launch_q0_1(const EmbedPlan &, EmbedParams &, cudaStream_t),
    embed_launch_q1_0(const EmbedPlan &, EmbedParams &, cudaStream_t), embed_launch_q1_1(const EmbedPlan &, EmbedParams &, cudaStream_t),
    embed_launch_q2_0(const EmbedPlan &, EmbedParams &, cudaStream_t), embed_launch_q2_1(const EmbedPlan &, EmbedParams &, cudaStream_t),
    embed_launch_q3_0(const EmbedPlan &, EmbedParams &, cudaStream_t), embed_launch_q3_1(const EmbedPlan &, EmbedParams &, cudaStream_t);
static const EmbedLaunch kLaunch[4][2] = {{embed_launch_q0_0, embed_launch_q0_1},
                                          {embed_launch_q1_0, embed_launch_q1_1},
                                          {embed_launch_q2_0, embed_launch_q2_1},
                                          {embed_launch_q3_0, embed_launch_q3_1}};
static_assert(SCONE_QUANT_FP16 == 0 && SCONE_QUANT_INT8 == 1 && SCONE_QUANT_INT4 == 2 && SCONE_QUANT_FP32 == 3 && SCONE_OUT_BF16 == 0 &&
                  SCONE_OUT_FP16 == 1,
              "kLaunch is indexed [quant][out_dtype]");

static int num_sms() {
    static int n = 0;
    if (n == 0) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
            n = kNumSMsB200;
    }
    return n;
}

// P = the fewest lanes per position the vocabulary needs; `resolved`: p.fgram_in holds the f-gram ids.
static int dispatch(int P, bool resolved, EmbedParams &p, int quant, int out_dtype, cudaStream_t stream) {
    const EmbedCall call{p.D, p.row_stride, p.pos != nullptr, p.additive != 0, resolved, P, getenv("SCONE_EMBED_PIPE"), p.T, num_sms()};
    const int rc = kLaunch[quant][out_dtype](plan_embed(call), p, stream);
    if (rc != SCONE_OK) return rc;
    SCONE_LAUNCHED();
    return SCONE_OK;
}

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
    p.group_shift = group_shift(t->group);
    return SCONE_OK;
}

// The argument checks and parameters the two matching entries share; `who` names the entry in the error messages.  p.T == 0
// on return: nothing to do.
static int matching_params(EmbedParams &p, const char *who, const scone_index_impl *ix, const void *d_base_emb, int64_t base_rows,
                           const void *d_pos_emb, const int64_t *d_ids, int64_t B, int64_t L, void *d_out, int32_t out_dtype,
                           int32_t *d_out_id, uint8_t *d_out_len, uint32_t *d_status) {
    SCONE_REQUIRE(out_dtype == SCONE_OUT_BF16 || out_dtype == SCONE_OUT_FP16, "%s: out_dtype must be bf16 or fp16", who);
    SCONE_REQUIRE(B >= 0 && L >= 0, "%s: negative shape", who);
    p.T = B * L;
    if (p.T == 0) return SCONE_OK;
    SCONE_REQUIRE(p.T < (1ll << 40), "%s: batch too large", who);
    SCONE_REQUIRE(d_ids && d_out, "%s: NULL ids or out", who);
    SCONE_REQUIRE(d_base_emb && base_rows > 0, "%s: base embedding table required (fallback rows)", who);
    SCONE_REQUIRE((((uintptr_t)d_base_emb | (uintptr_t)d_out | (uintptr_t)d_pos_emb) & 15) == 0,
                  "%s: base_emb, pos_emb and out must be 16-byte aligned", who);
    p.ix = view_of(ix, p.T);
    p.fgram_in = nullptr;
    p.base = static_cast<const uint8_t *>(d_base_emb);
    p.V = base_rows;
    p.pos = static_cast<const uint8_t *>(d_pos_emb);
    p.ids = d_ids;
    p.L = L;
    p.out = static_cast<uint8_t *>(d_out);
    p.out_id = d_out_id;
    p.out_len = d_out_len;
    p.status = d_status;
    return SCONE_OK;
}

}  // namespace scone

using namespace scone;

extern "C" {

static int embed_forward_impl(const scone_index_t *index, const scone_table_desc_t *table, const void *d_base_emb, int64_t base_rows,
                              const void *d_pos_emb, const int64_t *d_ids, int64_t B, int64_t L, void *d_out, int32_t out_dtype,
                              int32_t *d_out_id, uint8_t *d_out_len, uint32_t *d_status, void *stream_, uint32_t flags) {
    SCONE_REQUIRE(index && table, "scone_embed_forward: NULL index or table");
    const scone_index_impl *ix = reinterpret_cast<const scone_index_impl *>(index);
    EmbedParams p{};
    int rc = matching_params(p, "scone_embed_forward", ix, d_base_emb, base_rows, d_pos_emb, d_ids, B, L, d_out, out_dtype, d_out_id, d_out_len,
                             d_status);
    if (rc != SCONE_OK || p.T == 0) return rc;
    SCONE_REQUIRE(ix->n <= table->num_rows, "scone_embed_forward: index has %lld f-grams but the table only %lld rows",
                  (long long)ix->n, (long long)table->num_rows);
    rc = fill_table(p, table, "scone_embed_forward");
    if (rc != SCONE_OK) return rc;
    p.additive = (flags & SCONE_EMBED_ADDITIVE) ? 1 : 0;
    p.flags = flags;
    return dispatch(lanes_per_position(ix->len_mask, ix->max_n), false, p, table->quant, out_dtype, (cudaStream_t)stream_);
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
    SCONE_REQUIRE(index && shard && d_shard_rows, "scone_embed_forward_sharded: NULL index, shard descriptor or pointer table");
    SCONE_REQUIRE(world >= 1 && world <= 64, "scone_embed_forward_sharded: world %d outside [1, 64]", world);
    const scone_index_impl *ix = reinterpret_cast<const scone_index_impl *>(index);
    EmbedParams p{};
    int rc = matching_params(p, "scone_embed_forward_sharded", ix, d_base_emb, base_rows, d_pos_emb, d_ids, B, L, d_out, out_dtype, d_out_id,
                             d_out_len, d_status);
    if (rc != SCONE_OK || p.T == 0) return rc;
    SCONE_REQUIRE(ix->n <= total_rows, "scone_embed_forward_sharded: index has %lld f-grams but the shards only %lld rows", (long long)ix->n,
                  (long long)total_rows);
    SCONE_REQUIRE((total_rows + world - 1) / world <= shard->num_rows, "scone_embed_forward_sharded: %lld rows over %d shards exceed the shard capacity %lld",
                  (long long)total_rows, world, (long long)shard->num_rows);
    scone_table_desc_t geom = *shard;
    if (!geom.d_rows) geom.d_rows = reinterpret_cast<const void *>(uintptr_t(16));  // geometry only; never dereferenced when world > 1
    rc = fill_table(p, &geom, "scone_embed_forward_sharded");
    if (rc != SCONE_OK) return rc;
    p.shard_rows = reinterpret_cast<const uint8_t *const *>(d_shard_rows);
    p.rows = nullptr;
    p.num_rows = total_rows;
    p.world = -world;  // negative: always go through the pointer table, even for one shard
    return dispatch(lanes_per_position(ix->len_mask, ix->max_n), false, p, shard->quant, out_dtype, (cudaStream_t)stream_);
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
    return dispatch(4, true, p, table->quant, out_dtype, stream);
}

}  // extern "C"
