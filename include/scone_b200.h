/*
 * scone_b200.h -- C ABI of the B200-native SCONE input-embedding lookup.
 *
 * This is the drop-in boundary for ONE path of llmsresearch/scone: the
 * inference-time input-embedding lookup.  The reference has no FFI of its own
 * (it is pure Python); each entry point below names the reference interface
 * (file:line, relative to the upstream repository root) whose work it takes
 * over.  The Python mirror of the reference classes (scone_b200/tokenization,
 * scone_b200/inference) binds exactly these symbols through ctypes;
 * INTEGRATION.md shows the stub a reference maintainer would add.
 *
 * Conventions
 *   - plain C: pointers, sizes, opaque handles; no torch / C++ types.
 *   - every pointer named d_* is a DEVICE pointer (or a device-mapped pinned
 *     host pointer where stated) valid on the current CUDA device.
 *   - all work is enqueued asynchronously on `stream` (a cudaStream_t passed
 *     as void*); buffers must stay alive until the stream is synchronised.
 *     The only calls that synchronise are scone_index_create (one read-back of
 *     the build audit).
 *   - return value: 0 = OK, negative = error (SCONE_E_*); the message is
 *     available from scone_last_error() on the calling thread.
 *   - there is NO CPU fallback: without a CUDA device every compute entry
 *     point returns SCONE_E_CUDA.
 */
#ifndef SCONE_B200_H
#define SCONE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SCONE_B200_VERSION 200 /* 0.2.0 */

/* error codes */
#define SCONE_OK 0
#define SCONE_E_INVALID (-1) /* bad argument */
#define SCONE_E_CUDA (-2)    /* CUDA runtime error (incl. no device) */
#define SCONE_E_VOCAB (-3)   /* vocabulary rejected: duplicate key, bad length, negative token */
#define SCONE_E_NOMEM (-4)

/* cache-row storage formats (SURVEY.md section 8c; formulas in oracle/py_oracle.py) */
#define SCONE_QUANT_FP16 0 /* row = D x fp16                       (reference: `.half()`, scone/inference/engine.py:265-266) */
#define SCONE_QUANT_INT8 1 /* row = D x int8, then 1 x fp32 scale  (per-row symmetric) */
#define SCONE_QUANT_INT4 2 /* row = D/2 bytes (two nibbles q+8, element 2k low), then D/group x fp16 scales */
#define SCONE_QUANT_FP32 3 /* row = D x fp32, unquantised -- what the reference itself stores and returns
                              (scone/inference/embedding_cache.py:84-91, :99, :111, :132-135) */

/* output element types */
#define SCONE_OUT_BF16 0
#define SCONE_OUT_FP16 1
#define SCONE_OUT_FP32 2 /* only for scone_table_gather (the reference's fp32 get_embeddings) */

/* bits of the device status word written by scone_embed_forward */
#define SCONE_STATUS_TOKEN_OOR 1u /* a position with no f-gram had a token id outside [0, base_rows): row zero-filled
                                     (the reference raises IndexError from wte(), scone/models/language_model.py:239) */

#define SCONE_MAX_N 7 /* longest f-gram the 32-byte slot format holds */

typedef struct scone_index scone_index_t; /* opaque: device-resident f-gram index */

typedef struct scone_index_info {
    int64_t num_fgrams;
    int64_t capacity;    /* slots */
    int64_t bytes;       /* device bytes held by the handle */
    int32_t max_n;
    uint32_t len_mask;   /* bit (n-1) set when some f-gram has length n */
    int32_t max_probe;   /* longest insert probe sequence seen at build time */
    int32_t slot_bytes;  /* 32 for the wide format, 16 for compact-16 (every token < 65535, max_n <= 6) and compact-20
                            (every token < 1048575, max_n <= 5, fewer than 2^28 - 1 f-grams) */
    int64_t filter_bytes; /* bytes of the L2-resident pre-filter (included in `bytes`), 0 = none */
    int32_t slot_format;  /* 0 = 32-byte slots, 1 = compact 16-byte (six 16-bit tokens), 2 = compact 16-byte (five 20-bit tokens) */
    int32_t reserved;
} scone_index_info_t;

/* Where the cache rows live and how they are encoded.  Row r starts at
 * rows + r * row_stride; payload first, scales at byte `scale_offset`. */
typedef struct scone_table_desc {
    const void *d_rows;   /* device pointer, or device-mapped pinned host pointer (offloaded tier) */
    int64_t row_stride;   /* bytes; multiple of 16 */
    int64_t num_rows;     /* N; row index = f-gram id (scone/inference/embedding_cache.py:77,99) */
    int32_t quant;        /* SCONE_QUANT_* */
    int32_t dim;          /* D; multiple of 8 (INT4: multiple of group) */
    int32_t group;        /* INT4 group size (multiple of 8; 128 by default); ignored otherwise */
    int32_t scale_offset; /* byte offset of the scale(s) inside a row; ignored for FP16 */
} scone_table_desc_t;

/* ---- library ------------------------------------------------------------- */
int scone_version(void);
const char *scone_last_error(void);

/* ---- f-gram index ---------------------------------------------------------
 * Replaces the Python set/dict of int tuples held by NGramExtractor
 * (scone/tokenization/n_gram_extractor.py:41-44, filled at :96-99 / :159-165).
 *
 * d_tokens: int32 [n, max_n], f-gram r in row r in reading order, padded with -1.
 * d_lens  : uint8 [n].  The id of an f-gram is its row number (frequency rank in the
 *           reference, n_gram_extractor.py:98-99).
 * The open-addressing table (key stored inline, home slot from a rolling 64-bit hash)
 * is built by kernels on `stream`; the call then reads back a build audit and fails
 * with SCONE_E_VOCAB if two rows hold the same f-gram, a length is outside [1, max_n]
 * or a token is negative.  The slot format is compact-16 if it holds the vocabulary, else
 * compact-20 if it does, else wide:
 *   compact-16: 16 bytes, id + six 16-bit tokens: every token < 65535 and max_n <= 6;
 *   compact-20: 16 bytes, 28-bit id + five 20-bit tokens: every token < 1048575, max_n <= 5
 *               and fewer than 2^28 - 1 f-grams;
 *   wide:       32 bytes, id + seven int32 tokens: any vocabulary.
 * A probe step reads one 64-byte block: four compact slots or two wide ones.  load_factor in
 * (0, 0.9]; <= 0 -> 0.25 (128 B of index per f-gram with 32-byte slots, 64 B with 16-byte
 * slots): short probe chains matter more than index size, see DESIGN.md. */
int scone_index_create(const int32_t *d_tokens, const uint8_t *d_lens, int64_t n, int32_t max_n,
                       double load_factor, void *stream, scone_index_t **out);
int scone_index_destroy(scone_index_t *index);
int scone_index_info(const scone_index_t *index, scone_index_info_t *info);

/* Longest f-gram ENDING at every position (Algorithm 2, assets/algorithm.png; the
 * reference primitive is the membership test of n_gram_extractor.py:121-122 and the
 * tuple->id lookup of embedding_cache.py:173).  Rows of the [B, L] batch are independent;
 * pads are ordinary tokens (f_gram_tokenizer.py:122-123).
 * d_ids int64 [B, L] -> d_out_id int32 [B, L] (-1 = none), d_out_len uint8 [B, L] (0 = none). */
int scone_index_lookup(const scone_index_t *index, const int64_t *d_ids, int64_t B, int64_t L,
                       int32_t *d_out_id, uint8_t *d_out_len, void *stream);

/* d_out int32 [B, L, max_n]: id of the n-gram ending at position i (slot n-1), or -1.
 * This is the batched form of NGramExtractor.get_token_f_grams (n_gram_extractor.py:106-126):
 * the per-position "all f-grams containing the token" lists are a re-indexing of it. */
int scone_index_match_all(const scone_index_t *index, const int64_t *d_ids, int64_t B, int64_t L,
                          int32_t *d_out, void *stream);

/* NGramExtractor.fit on the device (scone/tokenization/n_gram_extractor.py:72-104): count every n-gram (n = 1..max_n, never
 * across texts) of a tokenised corpus, keep the max_f_grams most frequent (ties: first seen in the reference's enumeration
 * order text -> n -> start, :91), THEN drop counts below min_freq (:92-94); id = rank (:98-99).
 * d_tokens int32 [num_tokens] = the texts back to back, d_text_offsets int64 [num_texts + 1].  Output, in id order:
 * d_out_tokens int32 [max_f_grams, max_n] (-1 padded), d_out_lens uint8 [max_f_grams], optional d_out_counts int64; *out_n =
 * number of f-grams written, *out_distinct = distinct n-grams in the corpus (may be NULL).
 * n-gram occurrences are hashed (64 bits, `seed`), radix-sorted and run-length counted; every run is verified to hold a single
 * n-gram -- if two n-grams share a hash the call fails with SCONE_E_VOCAB and the caller retries with another seed.
 * Synchronises the stream (it returns counts); scratch is allocated with cudaMallocAsync (32 bytes per n-gram occurrence);
 * at most 2^31 - 1 occurrences per call. */
int scone_fit_vocab(const int32_t *d_tokens, int64_t num_tokens, const int64_t *d_text_offsets, int64_t num_texts,
                    int32_t max_n, int64_t min_freq, int64_t max_f_grams, uint64_t seed,
                    int32_t *d_out_tokens, uint8_t *d_out_lens, int64_t *d_out_counts,
                    int64_t *out_n, int64_t *out_distinct, void *stream);

/* ---- cache table ------------------------------------------------------------
 * Replaces EmbeddingCache's Dict[int, ndarray] / np.memmap [N, D] fp32 store
 * (scone/inference/embedding_cache.py:49-50, :76-91). */

/* Row geometry for a format: stride rounded up to `align` bytes (multiple of 16; 0 -> 32). */
int scone_table_layout(int32_t quant, int32_t dim, int32_t group, int32_t align,
                       int64_t *row_stride, int32_t *scale_offset);

/* cache_embeddings (embedding_cache.py:56-111): quantise k fp32 rows and store them at
 * table rows d_row_ids[0..k) (NULL -> rows row_base .. row_base+k).  d_rows_f32: float [k, D]. */
int scone_table_store(const scone_table_desc_t *table, const float *d_rows_f32, const int64_t *d_row_ids,
                      int64_t row_base, int64_t k, void *stream);

/* cache_embeddings with the reference's bias-free `f_gram_projection` (scone/models/language_model.py:172-176, applied at
 * :236 on every forward pass) folded into the table build:  table[row r] = quantise(d_rows[r, :] @ d_proj^T).
 * d_rows_bf16: bf16 [k, in_dim] (the f-gram model's output rows), d_proj_bf16: bf16 [dim, in_dim] (nn.Linear weight layout:
 * out_features x in_features), both row-major, 16-byte aligned, in_dim a multiple of 8; table->dim a multiple of 64.
 * A tcgen05 / TMEM GEMM (bf16 x bf16 -> fp32) whose epilogue IS the quantise-and-store of scone_table_store: the fp32
 * [k, dim] product is never written to memory.  Rows go to d_row_ids[0..k) (NULL -> row_base ..); destinations outside the
 * table are skipped and counted in *d_bad (may be NULL).  Result: the fp32 product of the bf16 inputs (fp32 accumulation in
 * tensor-core order) through exactly the quantiser of scone_table_store. */
int scone_table_store_projected(const scone_table_desc_t *table, const void *d_rows_bf16, const void *d_proj_bf16,
                                int32_t in_dim, const int64_t *d_row_ids, int64_t row_base, int64_t k,
                                uint32_t *d_bad, void *stream);

/* get_embeddings (embedding_cache.py:113-147): out[r] = dequant(table[d_row_ids[r]]) as
 * out_dtype ([k, D] contiguous).  Row ids outside [0, num_rows) produce a zero row and set
 * bit SCONE_STATUS_TOKEN_OOR in *d_status when d_status is not NULL. */
int scone_table_gather(const scone_table_desc_t *table, const int64_t *d_row_ids, int64_t k,
                       void *d_out, int32_t out_dtype, uint32_t *d_status, void *stream);

/* Raw copy of stored rows (no dequant): out[r, :] = the row_stride bytes of table row d_row_ids[r] (int32).
 * The owner-side step of the row-sharded tier: quantised bytes travel over NVLink and are dequantised by
 * the requester (scone_embed_gather on the received buffer).  d_out: [k, row_stride] bytes, 16-byte aligned. */
int scone_table_gather_packed(const scone_table_desc_t *table, const int32_t *d_row_ids, int64_t k,
                              void *d_out, uint32_t *d_status, void *stream);

/* ---- the fused hot path -----------------------------------------------------
 * One pass replacing, per position: get_token_f_grams + f_gram_to_id + get_embeddings
 * + the engine's assemble loop + the wte fallback
 * (n_gram_extractor.py:106-126, embedding_cache.py:149-181, engine.py:235-266,
 *  language_model.py:239-243), with Algorithm-2 semantics:
 *
 *   out[b, i, :] = dequant(table[fgram_id[b, i]])     if an f-gram ends at (b, i)
 *                = base_emb[ids[b, i], :]              otherwise
 *
 * d_base_emb : [base_rows, D] in out_dtype (bf16 / fp16), row stride D elements.
 * d_out      : [B, L, D] out_dtype, contiguous -- the transformer's inputs_embeds layout
 *              (language_model.py:257-258).
 * d_pos_emb  : optional [>= L, D] in out_dtype; when not NULL, pos_emb[i] is added (fp32 add,
 *              RNE) -- the wpe term of language_model.py:253-254.  NULL in the plain path.
 * d_out_id / d_out_len / d_status may be NULL. */
int scone_embed_forward(const scone_index_t *index, const scone_table_desc_t *table,
                        const void *d_base_emb, int64_t base_rows, const void *d_pos_emb,
                        const int64_t *d_ids, int64_t B, int64_t L,
                        void *d_out, int32_t out_dtype,
                        int32_t *d_out_id, uint8_t *d_out_len, uint32_t *d_status, void *stream);

/* Same kernel, reference-CODE combine instead of Algorithm 2's replace-or-fallback: the f-gram row is ADDED to the
 * token embedding, `combined_embeddings = base_embeddings + f_gram_embeddings` (scone/models/language_model.py:239-243),
 * with the row of the longest f-gram ending at the position as the f-gram term (zeros where none, engine.py:238):
 *
 *   out[b, i, :] = base_emb[ids[b, i], :] + dequant(table[fgram_id[b, i]])   if an f-gram ends at (b, i)
 *                = base_emb[ids[b, i], :]                                     otherwise
 *
 * (+ pos_emb[i] when d_pos_emb is not NULL; language_model.py:253-254).  All adds in fp32 in the reference's order
 * (base + row) + pos, ONE rounding (RNE) to out_dtype.  A token id outside [0, base_rows) contributes a zero base row
 * and sets SCONE_STATUS_TOKEN_OOR.  Arguments as scone_embed_forward. */
int scone_embed_forward_additive(const scone_index_t *index, const scone_table_desc_t *table,
                                 const void *d_base_emb, int64_t base_rows, const void *d_pos_emb,
                                 const int64_t *d_ids, int64_t B, int64_t L,
                                 void *d_out, int32_t out_dtype,
                                 int32_t *d_out_id, uint8_t *d_out_len, uint32_t *d_status, void *stream);

/* Options of the fused call (scone_embed_forward_ex); a NULL pointer means all defaults. */
#define SCONE_EMBED_ADDITIVE 1u      /* the combine of scone_embed_forward_additive */
#define SCONE_EMBED_INPUTS_STABLE 2u /* the caller vouches that NONE of this call's inputs (d_ids, the index, the table rows,
                                        d_base_emb, d_pos_emb) is written by the kernel that precedes it on `stream`
                                        (a serving loop: ids arrive by cudaMemcpyAsync, tables are static).  The kernel is
                                        launched with programmatic stream serialization either way; with this flag its
                                        matching and row fetches start under the previous kernel's tail and only its
                                        writes wait for that kernel to complete.  Results are identical. */
typedef struct scone_embed_opts {
    uint32_t flags; /* SCONE_EMBED_* */
    uint32_t reserved[3];
} scone_embed_opts_t;

/* scone_embed_forward / scone_embed_forward_additive with explicit options (same reference lines:
 * n_gram_extractor.py:106-126, embedding_cache.py:149-181, engine.py:235-266, language_model.py:239-243). */
int scone_embed_forward_ex(const scone_index_t *index, const scone_table_desc_t *table,
                           const void *d_base_emb, int64_t base_rows, const void *d_pos_emb,
                           const int64_t *d_ids, int64_t B, int64_t L,
                           void *d_out, int32_t out_dtype,
                           int32_t *d_out_id, uint8_t *d_out_len, uint32_t *d_status,
                           const scone_embed_opts_t *opts, void *stream);

/* Second half only: ids already resolved (used by the sharded and staged tiers).
 * d_fgram_id int32 [T] (-1 = fallback to base_emb[d_ids[t]]). */
int scone_embed_gather(const scone_table_desc_t *table, const void *d_base_emb, int64_t base_rows,
                       const void *d_pos_emb, int64_t L,
                       const int64_t *d_ids, const int32_t *d_fgram_id, int64_t T,
                       void *d_out, int32_t out_dtype, uint32_t *d_status, void *stream);

/* Optional mode reproducing the reference CODE instead of Algorithm 2 (SURVEY.md 0.2): the engine's assemble loop
 * (scone/inference/engine.py:235-259) -- out[b, i] = mean of dequant(row) over ALL f-grams that CONTAIN position i
 * (list order of get_token_f_grams, n_gram_extractor.py:119-124: n ascending, then start ascending; fp32 sum in that
 * order, divided by the count), ZEROS where there is none.  No fallback row, no replacement: the reference adds this
 * (projected) tensor to wte(input_ids) afterwards (language_model.py:236-243).
 * d_work: int32 [B, L, max_n] scratch (filled with scone_index_match_all's result).  out_dtype may be FP32. */
int scone_embed_mean_forward(const scone_index_t *index, const scone_table_desc_t *table,
                             const int64_t *d_ids, int64_t B, int64_t L, int32_t *d_work,
                             void *d_out, int32_t out_dtype, void *stream);

/* Row-sharded table read DIRECTLY over NVLink (peer memory), fused into the same kernel: f-gram id r lives on rank
 * r % world, at row r / world of that rank's shard.  d_shard_rows is a DEVICE array of `world` pointers to the
 * shards as mapped into THIS process (peer-mapped allocations, e.g. torch symmetric-memory buffer_ptrs; entry
 * `rank` is the local shard).  `shard` describes the common row geometry (row_stride, quant, dim, ...; its d_rows is
 * ignored, its num_rows is the capacity of one shard); total_rows = number of f-gram rows over all shards.
 * The matcher warps turn (owner, local row) into a peer address and the TMA bulk copy / vector loads fetch the still
 * quantised row across NVSwitch straight into shared memory; no request/reply exchange, no host synchronisation, and
 * misses never leave the GPU.  Everything else is scone_embed_forward. */
int scone_embed_forward_sharded(const scone_index_t *index, const scone_table_desc_t *shard,
                                const void *const *d_shard_rows, int32_t world, int64_t total_rows,
                                const void *d_base_emb, int64_t base_rows, const void *d_pos_emb,
                                const int64_t *d_ids, int64_t B, int64_t L,
                                void *d_out, int32_t out_dtype,
                                int32_t *d_out_id, uint8_t *d_out_len, uint32_t *d_status, void *stream);

/* Offloaded tier: host memory for a table the GPU reads in place (the role of the reference's np.memmap backing store,
 * scone/inference/embedding_cache.py:76-91).  An anonymous mapping on transparent huge pages, first-touched by `nthreads`
 * host threads, registered with the driver as mapped + portable pinned memory.  *out_device is the pointer to put into
 * scone_table_desc_t.d_rows.  Release with scone_host_free(host pointer, same byte count). */
int scone_host_alloc(int64_t bytes, int32_t nthreads, void **out_host, void **out_device);
int scone_host_free(void *host, int64_t bytes);

/* Offloaded tier, STAGED variant (host code, no GPU work): copy rows h_row_ids[0..k) of a host-resident table into a
 * contiguous pinned staging buffer with `nthreads` host threads, ready for one cudaMemcpyAsync.  The zero-copy
 * variant needs nothing special: point scone_table_desc_t.d_rows at the pinned (UVA-mapped) table.
 * Returns SCONE_E_INVALID if an id is outside [0, num_rows). */
int scone_host_gather_rows(const void *h_rows, int64_t row_stride, int64_t num_rows, const int32_t *h_row_ids,
                           int64_t k, void *h_staging, int32_t nthreads);

/* ---- host-fed pipeline ----------------------------------------------------------------------------------
 * The throughput form of scone_embed_forward for callers whose ids live in HOST memory (the reference's engine
 * tokenises on the host, scone/inference/engine.py:222-233): `slots` batches rotate through the streams owned by
 * the pipeline -- copy-in (pinned host ids -> HBM), compute (the fused kernel), copy-out (match result -> pinned
 * host) -- chained per slot with events, so batch k+1's H2D and batch k-1's D2H run under batch k's kernel.
 * All buffers are the caller's: per slot d_ids int64 [B*L], d_out [B*L*D] out_dtype, d_meta / h_meta 5*B*L bytes
 * (fgram_id int32 [B*L] followed by match_len uint8 [B*L]; h_meta pinned).  The embeddings stay on the device. */
typedef struct scone_pipeline scone_pipeline_t;
int scone_pipeline_create(const scone_index_t *index, const scone_table_desc_t *table, const void *d_base_emb,
                          int64_t base_rows, const void *d_pos_emb, int64_t B, int64_t L, int32_t out_dtype,
                          int32_t slots, void *const *d_ids_slots, void *const *d_out_slots, void *const *d_meta_slots,
                          void *const *h_meta_slots, uint32_t *d_status, scone_pipeline_t **out);
/* Enqueue one batch from pinned host ids; *slot receives the slot it went to.  If that slot's previous batch has not
 * been waited for yet, the call waits for it first.  Returns without waiting for the new batch: h_ids_pinned is read by an
 * asynchronous copy and must stay untouched until scone_pipeline_wait(slot) has returned. */
int scone_pipeline_submit(scone_pipeline_t *p, const int64_t *h_ids_pinned, int32_t *slot);
/* The pipeline runs on streams of its own (copy-in, two alternating compute streams, copy-out), ordered against the caller only at creation.  After changing anything
 * the pipeline reads (table rows, base / position embeddings) on `stream`, call this before the next submit: every batch
 * submitted afterwards runs behind the work already enqueued on `stream`. */
int scone_pipeline_follow(scone_pipeline_t *p, void *stream);
/* Block the calling host thread until the batch in `slot` is complete: its embeddings are in d_out_slots[slot] and
 * its match result in h_meta_slots[slot]. */
int scone_pipeline_wait(scone_pipeline_t *p, int32_t slot);
int scone_pipeline_destroy(scone_pipeline_t *p);

/* Number of kernels this library has launched from the calling process (monotonic). */
int64_t scone_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* SCONE_B200_H */
