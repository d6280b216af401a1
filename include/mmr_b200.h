/*
 * mmr_b200.h -- C ABI of the B200-native exact-scan library (libmmr_b200.so).
 *
 * Drop-in boundary for ONE path of Sabarna07-tech/Multimodal-RAG-for-Image-Text-Search: the flat cosine
 * nearest-neighbour scan + top-k + text/image fusion + confidence gate behind retrieve_text /
 * retrieve_images.  The reference has no FFI of its own (it is 100 % Python; the arithmetic lives in the
 * third-party lancedb/lance Rust crate), so every entry point below cites the reference Python interface
 * it replaces.  The reference-side binding (a ctypes stub) is shown in INTEGRATION.md; the shipped host
 * mirror is multimodal-rag-for-image-text-search_b200/store.py (class B200Store == LanceDBStore's duck type).
 *
 * Conventions
 *   - extern "C", plain pointers and sizes; no C++ or torch types.  Every function returns an int status
 *     (MMR_OK == 0); mmr_last_error() gives a thread-local message.  No exception crosses the ABI.
 *   - Pointers named *_dev are device pointers on the index's device, *_host are host pointers.
 *   - The caller owns every buffer it passes (rows, queries, outputs, workspace); the library owns only
 *     the opaque index handle (segment table, device attributes, small staging buffers).
 *   - Every call that launches work takes the cudaStream_t to launch on (as void*) and is asynchronous
 *     with respect to the host unless documented otherwise.
 *   - There is no CPU fallback: on a machine without an sm_100 device the calls fail with MMR_ERR_CUDA.
 *   - Rows are ordinals into one resident index (< 2^32 rows per GPU); results carry int64 global row ids
 *     (ordinal + row_base of the shard).  Result order everywhere: score descending, row id ascending.
 */
#ifndef MMR_B200_H_
#define MMR_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MMR_ABI_VERSION 2

enum mmr_status {
  MMR_OK = 0,
  MMR_ERR_INVALID = 1,     /* bad argument */
  MMR_ERR_CUDA = 2,        /* CUDA runtime / driver error, or no usable sm_100 device */
  MMR_ERR_UNSUPPORTED = 3, /* valid request this build has no kernel for (e.g. dim not 384/512) */
  MMR_ERR_WORKSPACE = 4    /* workspace too small */
};

enum mmr_dtype {
  MMR_BF16 = 0, /* resident storage chosen by the north star */
  MMR_F32 = 1,  /* the reference's stored precision (list<float32>) */
  MMR_F16 = 2
};

enum mmr_query_precision {
  MMR_QP_AUTO = 0, /* batches of >= 3 queries on one row range run on the tensor cores with 16-bit queries */
  MMR_QP_F32 = 1,  /* every query is scored in fp32 (K1 family): a request's result is independent of its batch */
  MMR_QP_RESCORE = 2 /* batches of >= 3 on one row range: the tensor cores nominate 32 / 64 candidates per query, which are
                      * re-scored with the fp32 query in K1's arithmetic; the top-k is proven equal to K1's (else that
                      * query is rerun on K1), so results are bit-identical to single-query searches.  The call
                      * synchronises the stream once. */
};

#define MMR_MAX_K 64 /* INDEX_TOPK_TEXT defaults to 50, INDEX_TOPK_IMG to 12 (reference config.py:46-47) */

typedef struct mmr_index mmr_index;

/* Library / error plumbing. */
int mmr_abi_version(void);
const char* mmr_last_error(void);
/* Switches (DESIGN.md 6a: MMR_PDL, MMR_INLINE_QUERY, MMR_MAILBOX, MMR_ENC_FUSE_LN, MMR_ENC_ATT_MMA, MMR_ENC_GEMM_SMEM_KB,
 * MMR_ENC_NARROW_TILES; all but MMR_PDL are measurement switches whose defaults are the shipped path).  The
 * environment is read once when the library is loaded; these change / read a switch afterwards (value NULL or "" =
 * default).  mmr_get_option returns -1 for an unknown name. */
int mmr_set_option(const char* name, const char* value);
int mmr_get_option(const char* name);

/*
 * Resident index over caller-owned device rows.
 *   rows_dev        row-major [n_rows, dim] of `dtype`, 16-byte aligned, rows already L2-normalised
 *                   (what LanceDBStore._prepare_rows writes, app/storage/lancedb_store.py:71-85).
 *   seg_offsets_host  [n_segments + 1] ascending row offsets; segment t = rows [off[t], off[t+1]) = the
 *                   rows of one tenant.  Replaces the per-query `user_id == '...'` filter
 *                   (lancedb_store.py:107,118,141-144) with prefilter semantics.  NULL / 0 = one segment.
 *   row_base        added to every row id written out (row-range shard of a larger table).
 */
int mmr_index_create(int device, int dim, int dtype, int64_t n_rows, const void* rows_dev,
                     const int64_t* seg_offsets_host, int32_t n_segments, int64_t row_base, mmr_index** out);
int mmr_index_destroy(mmr_index* index);
/* Query precision policy of this index (enum mmr_query_precision).  The serving store sets MMR_QP_F32 so that what a
 * request gets never depends on which other requests shared its launch (the reference answers every request alone,
 * app/ml/retrieve.py:103-117). */
int mmr_index_set_query_precision(mmr_index* index, int mode);
/* Re-point an existing handle at grown / rewritten rows after an upsert (same dim and dtype). */
int mmr_index_update(mmr_index* index, int64_t n_rows, const void* rows_dev, const int64_t* seg_offsets_host,
                     int32_t n_segments);

/*
 * Loader (L1): fp32 embedding rows -> resident rows of `dtype`, optionally re-normalised exactly like
 * LanceDBStore._normalize (lancedb_store.py:63-69).  src and dst are device pointers.
 */
int mmr_convert_rows_f32(const float* src_dev, void* dst_dev, int dtype, int64_t n_rows, int dim, int normalize,
                         void* stream);
/* Same from pageable or pinned HOST memory, streamed through a double-buffered pinned staging area. */
int mmr_load_rows_f32_host(int device, const float* src_host, void* dst_dev, int dtype, int64_t n_rows, int dim,
                           int normalize, void* stream);

/* Same, with a row map: source row i is written to resident row dst_row_host[i]; negative entries are skipped.  This is
 * how the store uploads a host block in insertion order straight into its tenant-sorted place (the tenant grouping that
 * replaces the `user_id == '...'` filter, lancedb_store.py:107,118) without gathering 20 GB on the host.  NULL = identity.
 * dst_dev is the BASE of the resident matrix in this form. */
int mmr_load_rows_f32_host_scatter(int device, const float* src_host, void* dst_dev, int dtype, int64_t n_rows, int dim,
                                   int normalize, const int64_t* dst_row_host, void* stream);
/* Host-only helper of the columnar store: 64-bit hashes of n strings held Arrow-style (byte buffer + n+1 int32 offsets),
 * used to find the rows an upsert replaces (delete-by-chunk_id, lancedb_store.py:91-92). */
int mmr_hash_strings(const uint8_t* data, const int32_t* offsets, int64_t n, uint64_t* out);

/*
 * The scan: LanceDBStore.search_text / search_image (lancedb_store.py:103-123) for a batch of B queries.
 *   queries_dev     [B, dim] float32, any norm (re-normalised on device as :104 / :115 do).
 *   query_seg_host  [B] segment id per query, or NULL = every query scans the whole index; -1 = whole index.
 *   k               max(top_k, 1) of the reference; 1..MMR_MAX_K.
 *   out_scores_dev  [B, k] float32 cosine similarity, best first; -inf where fewer than k rows exist.
 *   out_rows_dev    [B, k] int64 row ids, -1 padded.
 *   workspace_dev   >= mmr_search_workspace_bytes(index, B, k) bytes, ZEROED once before its first use
 *                   (the library leaves it reusable); not shared between concurrently running searches.
 */
size_t mmr_search_workspace_bytes(const mmr_index* index, int32_t B, int32_t k);
/* Exact size for mmr_search_ranges with n_ranges row ranges in total (mmr_search_workspace_bytes budgets 8 per query). */
size_t mmr_search_ranges_workspace_bytes(const mmr_index* index, int32_t B, int32_t k, int64_t n_ranges);
int mmr_search(const mmr_index* index, const float* queries_dev, const int32_t* query_seg_host, int32_t B,
               int32_t k, float* out_scores_dev, int64_t* out_rows_dev, void* workspace_dev, size_t workspace_bytes,
               void* stream);
/*
 * Same scan with explicit row ranges per query instead of one segment id: query b scans
 * ranges_host[2*r], ranges_host[2*r+1]) for r in [range_off_host[b], range_off_host[b+1]).  This is how a store that
 * appends delta segments between compactions (upsert = tombstone + append, lancedb_store.py:87-101) searches a tenant
 * that currently owns several ranges.  Rows overwritten with NaN (tombstones) never appear in results.  The ranges of
 * one query must not overlap (MMR_ERR_INVALID).  Queries with identical range lists (the same tenant) are grouped four at
 * a time and share one pass over those rows (K6); every score is computed in fp32 exactly as for a single query.
 */
int mmr_search_ranges(const mmr_index* index, const float* queries_dev, int32_t B, int32_t k,
                      const int32_t* range_off_host, const int64_t* ranges_host, float* out_scores_dev,
                      int64_t* out_rows_dev, void* workspace_dev, size_t workspace_bytes, void* stream);
/*
 * Same with HOST buffers; this is the call B200Store.search_* makes per request and its time is the end-to-end figure in
 * bench.py.  Re-entrant (calls on one index take turns on its staging set).  For one or two queries on one row range the
 * query travels in the kernel's parameters and the kernel writes the result and a completion flag into a mapped pinned
 * mailbox the host spins on: one launch, no copies, no stream synchronisation.  Larger batches stage the queries with one
 * H2D copy, the kernels still write into the mailbox, and the stream is synchronised.
 */
int mmr_search_host(mmr_index* index, const float* queries_host, const int32_t* query_seg_host, int32_t B,
                    int32_t k, float* out_scores_host, int64_t* out_rows_host, void* stream);

/*
 * Cross-shard merge (K4): G shard-local results [G, B, k] -> [B, k].  Used after the all-gather when the
 * index is row-range sharded over GPUs; identical output for every G.
 */
int mmr_merge_topk(const float* scores_dev, const int64_t* rows_dev, int32_t G, int32_t B, int32_t k,
                   float* out_scores_dev, int64_t* out_rows_dev, void* stream);
/* Same, shard g's [B, k] block starting at element g * stride of each array: lets the merge read the
 * all-gathered wire buffer ([G][scores | rows]) in place. */
int mmr_merge_topk_strided(const float* scores_dev, const int64_t* rows_dev, int64_t score_shard_stride,
                           int64_t row_shard_stride, int32_t G, int32_t B, int32_t k, float* out_scores_dev,
                           int64_t* out_rows_dev, void* stream);

/*
 * Fused scan + exchange for row-range shards on one NVLink/NVSwitch box (replaces scan -> NCCL all-gather -> merge).
 * Every rank owns a symmetric buffer of mmr_exchange_buffer_bytes(G, B, k) bytes, ZEROED once, mapped into every
 * process (e.g. torch.distributed._symmetric_memory); peer_bufs_host[g] is rank g's buffer address as mapped in THIS
 * process.  Per search: the shard scan writes its [B, k] result straight into every peer's buffer with peer-mapped
 * stores and releases a flag (for B <= 2 inside the scan kernel's last CTA; otherwise a small push kernel), then a
 * wait+merge kernel acquires the G flags and merges the G lists.  seq = 1, 2, 3, ... identical on all ranks.
 * The answer equals mmr_search + all-gather + mmr_merge_topk bit for bit.  A peer that never arrives makes the merge
 * give up after 5 s and write row id -2 into out_rows[q * k] instead of hanging the GPU.
 */
size_t mmr_exchange_buffer_bytes(int32_t G, int32_t B, int32_t k);
size_t mmr_search_exchange_workspace_bytes(const mmr_index* index, int32_t B, int32_t k);
int mmr_search_exchange(const mmr_index* index, const float* queries_dev, const int32_t* query_seg_host, int32_t B,
                        int32_t k, const uint64_t* peer_bufs_host, int32_t G, int32_t rank, uint32_t seq,
                        float* out_scores_dev, int64_t* out_rows_dev, void* workspace_dev, size_t workspace_bytes,
                        void* stream);

/* The same exchange with HOST buffers, for one process per GPU: for B <= 2 the query rides in the scan kernel's
 * parameters, the wait+merge kernel writes the merged result and a completion flag into the index's mapped mailbox and
 * the host spins on it (no H2D / D2H copies, no stream synchronisation on the request path). */
int mmr_search_exchange_host(mmr_index* index, const float* queries_host, const int32_t* query_seg_host, int32_t B,
                             int32_t k, const uint64_t* peer_bufs_host, int32_t G, int32_t rank, uint32_t seq,
                             float* out_scores_host, int64_t* out_rows_host, void* stream);

/*
 * One process, G GPUs: the shape of the reference's deployment (ONE store object in ONE process, app/ml/retrieve.py:21)
 * on a multi-GPU box.  `shards[g]` is a row-range shard on its own device (row_base = its first global row; shard 0's
 * device collects).  A search runs one scan launch per device from per-device launcher threads; every scan kernel stores
 * its [B, k] result into the collector's exchange buffer over NVLink peer mappings, the collector's wait+merge kernel
 * writes the merged result and a completion flag into a mapped host mailbox.  Ranges are GLOBAL row ranges
 * (mmr_search_ranges convention); each shard scans its slice of them.  Results equal the single-GPU scan bit for bit.
 */
typedef struct mmr_multi mmr_multi;
int mmr_multi_create(mmr_index** shards, int32_t G, mmr_multi** out);
int mmr_multi_destroy(mmr_multi* multi);
int mmr_multi_search_host(mmr_multi* multi, const float* queries_host, int32_t B, int32_t k,
                          const int32_t* range_off_host, const int64_t* ranges_host, float* out_scores_host,
                          int64_t* out_rows_host);

/*
 * Fusion + gate (K5): _fuse_results with no rerank scores (reference app/ml/retrieve.py:158-195) and
 * _confidence_low (app/ml/generate.py:56-60), bit-identical float64 results.
 *   text_* [B, kt], img_* [B, ki] as written by mmr_search (either may be NULL with k = 0).
 *   out_combined [B, final_n] f64 combined (z) score; out_score [B, final_n] f64 the item's `score`;
 *   out_rows [B, final_n] i64 (-1 padded); out_modality [B, final_n] i8 (0 text, 1 image, -1 none);
 *   out_low_conf [B] u8.
 */
int mmr_fuse(const float* text_scores_dev, const int64_t* text_rows_dev, int32_t kt, const float* img_scores_dev,
             const int64_t* img_rows_dev, int32_t ki, int32_t B, int32_t final_n, double tau,
             double* out_combined_dev, double* out_score_dev, int64_t* out_rows_dev, int8_t* out_modality_dev,
             uint8_t* out_low_conf_dev, void* stream);

/*
 * Fusion + gate, complete form: _rerank_text's re-ordering (reference app/ml/retrieve.py:150-154), _fuse_results
 * (:158-183, including the rerank z-scores and their positional indexing), _z_scores (:186-195) and _confidence_low
 * (app/ml/generate.py:56-60), from the float64 scores the reference's Python sees.  The cross-encoder itself stays on
 * the host: its logits come in as text_rerank_dev, assigned to the first rerank_count[b] text items exactly as
 * `zip(top_candidates, scores)` assigns them (rerank_count_dev NULL = rerank off).  Bit-identical to the reference's own
 * outputs on the golden vectors (tests/golden/fusion_golden.json).
 *   text_scores [B, kt] scan order, text_count [B]; img_scores [B, ki], img_count [B];
 *   out_combined [B, final_n] f64; out_index [B, final_n] i32: text item j -> j, image item j -> kt + j, -1 = none.
 */
int mmr_fuse_f64(const double* text_scores_dev, const int32_t* text_count_dev, const double* text_rerank_dev,
                 const int32_t* rerank_count_dev, const double* img_scores_dev, const int32_t* img_count_dev,
                 int32_t kt, int32_t ki, int32_t B, int32_t final_n, double tau, double* out_combined_dev,
                 int32_t* out_index_dev, uint8_t* out_low_conf_dev, void* stream);

/*
 * Query encoders on the device (SURVEY 8f rank 2 / 3): the models in front of and behind the scan, so that a query is
 * born on the GPU and its embedding feeds mmr_search without a host hop.
 *   MMR_ENC_MINILM     embed_text_batch: MiniLM-L6 (BERT, post-LN), masked mean pooling, L2 norm -> [B, hidden]
 *                      (reference app/ml/embeddings.py:52-70, sentence-transformers/all-MiniLM-L6-v2)
 *   MMR_ENC_CLIP_TEXT  embed_query_for_images: CLIP text tower (pre-LN, causal), hidden state at the EOS token -> final
 *                      LayerNorm -> text_projection -> L2 norm -> [B, proj_dim]   (app/ml/embeddings.py:94-105)
 *   MMR_ENC_CROSS      CrossEncoder.predict: the same BERT + pooler (tanh) + 1-logit classifier -> [B] raw logits
 *                      (app/ml/retrieve.py:29-38,146; cross-encoder/ms-marco-MiniLM-L-6-v2)
 *   MMR_ENC_CLIP_VISION  embed_images_batch, the ingest side: CLIP vision tower (ViT-B/32) -> [B, proj_dim]
 *                      (app/ml/embeddings.py:73-91); created with mmr_encoder_create_vision, run with
 *                      mmr_encoder_forward_pixels (below)
 * Tokenisation stays with the caller (HF tokenizers need the vocabulary files): the calls take token ids.
 * Weights are handed over once, by name, as fp32 device arrays in nn.Linear layout ([out, in]); GEMM weights are kept
 * as bf16, everything else as fp32:
 *   word_emb pos_emb type_emb emb_ln_w emb_ln_b | L<i>.qkv_w ([3H, H]: q, k, v stacked) L<i>.qkv_b L<i>.o_w L<i>.o_b
 *   L<i>.ln1_w L<i>.ln1_b L<i>.fc1_w L<i>.fc1_b L<i>.fc2_w L<i>.fc2_b L<i>.ln2_w L<i>.ln2_b | final_ln_w final_ln_b proj_w
 *   (CLIP) | pooler_w pooler_b cls_w cls_b (cross-encoder).  ln1 / ln2 are the first / second LayerNorm of a layer.
 */
enum mmr_encoder_kind { MMR_ENC_MINILM = 0, MMR_ENC_CLIP_TEXT = 1, MMR_ENC_CROSS = 2 };
typedef struct mmr_encoder_config {
  int32_t kind;           /* enum mmr_encoder_kind */
  int32_t vocab_size;
  int32_t hidden;         /* 384 (MiniLM) or 512 (CLIP) */
  int32_t layers;
  int32_t heads;          /* head dim 32 or 64 */
  int32_t intermediate;   /* multiple of 128 */
  int32_t max_positions;
  int32_t type_vocab;     /* BERT token types (2); ignored for CLIP */
  int32_t proj_dim;       /* CLIP text_projection rows; ignored otherwise */
  int32_t eos_token_id;   /* CLIP pooling position (first occurrence; 2 = legacy argmax rule) */
  float ln_eps;
} mmr_encoder_config;
typedef struct mmr_encoder mmr_encoder;
int mmr_encoder_create(int device, const mmr_encoder_config* config, mmr_encoder** out);
int mmr_encoder_destroy(mmr_encoder* encoder);
int mmr_encoder_out_dim(const mmr_encoder* encoder);
int mmr_encoder_set_weight(mmr_encoder* encoder, const char* name, const float* data_dev, int64_t numel, void* stream);
/* One forward pass for B sequences padded to S tokens.  S <= 512, except S <= 330 for a model with head dim 64 whose
 * attention runs on the fp32 kernel: the query encoders (MMR_ENC_MINILM, MMR_ENC_CLIP_TEXT) unless MMR_ENC_ATT_MMA=2 (the
 * cross-encoder's tensor-core attention takes 512 at either head dim).  Longer sequences fail with MMR_ERR_UNSUPPORTED.
 * ids / mask (1 = token, 0 = padding; NULL = all ones) /
 * token types (NULL = all zero) are HOST arrays [B, S]; out_dev is [B, out_dim] fp32 on the encoder's device
 * (L2-normalised embeddings, or [B] logits for MMR_ENC_CROSS) -- directly usable as mmr_search's queries_dev. */
int mmr_encoder_forward(mmr_encoder* encoder, const int32_t* input_ids_host, const int32_t* attention_mask_host,
                        const int32_t* token_type_host, int32_t B, int32_t S, float* out_dev, void* stream);

/*
 * CLIP vision tower (HF CLIPVisionModelWithProjection; what CLIPModel.get_image_features computes): pixels -> patch
 * embedding (Conv2d, stride = kernel = patch_size, no bias, run as patchify + one GEMM) -> class token + position
 * embeddings -> pre-LayerNorm -> `layers` pre-LN quick-GELU layers (no mask, not causal) -> class token -> final LayerNorm
 * (HF post_layernorm) -> visual_projection -> L2 norm.  Image preprocessing (decode, resize, crop, normalise) stays with the
 * caller (HF CLIPImageProcessor), as tokenisation does for the text encoders.
 * Config limits, checked before any CUDA call (MMR_ERR_INVALID / MMR_ERR_UNSUPPORTED with a message): hidden 768 with head
 * dim 64; image_size a multiple of patch_size; channels * patch_size^2 a multiple of 64; intermediate a multiple of 128;
 * (image_size / patch_size)^2 + 1 <= 330 tokens (the fp32 attention at head dim 64: ViT-B/32 has 50, ViT-B/16 197);
 * 0 < proj_dim <= hidden.
 * Weights by name through mmr_encoder_set_weight: patch_w ([hidden, channels * patch_size^2]: the Conv2d weight
 * [hidden, C, P, P] flattened, kept as bf16) cls_emb ([hidden]) pos_emb ([tokens, hidden]) pre_ln_w pre_ln_b |
 * L<i>.* exactly as for MMR_ENC_CLIP_TEXT | final_ln_w final_ln_b proj_w ([proj_dim, hidden]).
 * mmr_encoder_forward on a vision encoder, and mmr_encoder_forward_pixels on a text encoder, fail with MMR_ERR_INVALID.
 */
enum { MMR_ENC_CLIP_VISION = 3 };
typedef struct mmr_vision_config {
  int32_t hidden, layers, heads, intermediate, image_size, patch_size, channels, proj_dim;
  float ln_eps;
} mmr_vision_config;
int mmr_encoder_create_vision(int device, const mmr_vision_config* config, mmr_encoder** out);
/* One forward pass for B >= 1 images: pixels_dev fp32 [B, channels, image_size, image_size] (NCHW, what
 * CLIPImageProcessor returns) on the encoder's device; out_dev [B, proj_dim] fp32 unit-norm rows, directly usable as
 * mmr_search queries or as rows for mmr_convert_rows_f32.  Calls on one encoder take turns, as mmr_encoder_forward's do. */
int mmr_encoder_forward_pixels(mmr_encoder* encoder, const float* pixels_dev, int32_t B, float* out_dev, void* stream);

/*
 * CLIP image preprocessing on the device, in front of mmr_encoder_forward_pixels: B decoded 8-bit RGB images of any sizes
 * -> out_dev fp32 [B, 3, crop_h, crop_w] (NCHW), bit-identical to Pillow's Image.resize((out_w, out_h), BICUBIC) followed
 * by a crop at (top, left) and the per-channel map table[c][byte] (HF CLIPImageProcessorPil: resize, centre crop, rescale,
 * normalise; the caller computes the geometry and builds the table with HF's own rescale / normalise).
 *   src_dev    the images, packed HWC RGB (3 bytes per pixel, rows contiguous), each starting at a multiple of 16 bytes
 *              from a 16-byte aligned src_dev; the kernel reads whole 16-byte words, so each image's bytes rounded up to
 *              a multiple of 16 must lie within src_bytes
 *   geom_host  HOST array [B][7]: offset (bytes into src_dev), h, w, out_h, out_w (the resized size), top, left (the crop
 *              window's origin in the resized image)
 * Limits, checked with every other argument before any CUDA call (MMR_ERR_INVALID with a message): 1 <= crop_h, crop_w <=
 * MMR_PREP_MAX_CROP; 1 <= h, w <= MMR_PREP_MAX_SIDE; 1 <= out_h, out_w <= MMR_PREP_MAX_OUT; top, left >= 0 with
 * top + crop_h <= out_h and left + crop_w <= out_w; a downscale of at most 63.5x per axis (Pillow's bicubic window of
 * 2 * ceil(2 * in / out) + 1 taps <= MMR_PREP_MAX_TAPS).  One launch per MMR_PREP_LAUNCH_IMAGES images, on `stream`.
 */
enum { MMR_PREP_MAX_CROP = 4096, MMR_PREP_MAX_SIDE = 65535, MMR_PREP_MAX_OUT = 1 << 24, MMR_PREP_MAX_TAPS = 255,
       MMR_PREP_LAUNCH_IMAGES = 896 };
typedef struct mmr_image_prep {
  int32_t crop_h, crop_w;
  float table[3][256];   /* pixel_values[c] = table[c][resized byte of channel c] */
} mmr_image_prep;
int mmr_image_preprocess(int device, const mmr_image_prep* cfg, const uint8_t* src_dev, int64_t src_bytes, const int64_t* geom_host,
                         int32_t B, float* out_dev, void* stream);

/*
 * Validation hook for the tensor-core path (K2): raw cosine scores of B queries against rows
 * [row_begin, row_end) as computed by the tcgen05 contraction (bf16 queries x bf16 rows, fp32 accumulate),
 * written to out_scores_dev[b * out_ld + (row - row_begin)].  workspace as for mmr_search(B, k = 10).
 */
int mmr_debug_umma_scores(const mmr_index* index, const float* queries_dev, int32_t B, int64_t row_begin,
                          int64_t row_end, float* out_scores_dev, int64_t out_ld, void* workspace_dev,
                          size_t workspace_bytes, void* stream);

/*
 * Validation hooks for the encoder kernels: each runs ONE launch of the kernel the forward pass runs, through the same
 * launch code, on caller-owned device buffers (row-major).  Arguments are checked before any CUDA call (MMR_ERR_INVALID
 * with a message).
 *   mmr_debug_enc_gemm       gemm_wt_kernel: out[t, f] = epilogue(sum_k X[t, k] W[f, k] + bias[f]), t < M, f < N.
 *       epi       0 out_f32 = y; 1 out_f32 = y + residual (residual may equal out_f32: the in-place residual stream);
 *                 2 out_bf16 = GELU(erf)(y); 3 out_bf16 = quick-GELU(y)
 *       nt        token tile 64, 128 or 256 (box rows of X's tensor map)
 *       fold_ln   0: x_dev is X bf16 [M, K].  1: X = bf16(LayerNorm(ln_src_dev fp32 [M, K]; ln_g, ln_b, ln_eps)) computed
 *                 inside the GEMM (nt 64, K 384 or 512, epi != 1), the normalised rows also written to ln_out_dev fp32 [M, K]
 *                 when it is not NULL (must not alias ln_src)
 *       W bf16 [N, K]; N a multiple of 128, K of 64; bias fp32 [N] or NULL; residual / out_f32 fp32 [M, N]; out_bf16 bf16 [M, N]
 *   mmr_debug_enc_attention  softmax(q k^T / sqrt(H / heads)) v per (sequence, head) over qkv fp32 [B * S, 3H] (q | k | v)
 *       -> ctx bf16 [B * S, H]; tensor_cores 1 = attention_mma_kernel, 0 = attention_kernel; mask int32 [B * S] (0 = padding
 *       key) or NULL; causal hides keys after the query row.  Sequence limits as for mmr_encoder_forward.
 *   mmr_debug_enc_layernorm  layernorm_kernel<H>, H 384 or 512: rows of x fp32 [M, H] -> out_f32 (may equal x) and / or
 *       out_bf16 bf16 [M, H].
 *   mmr_debug_enc_patch_embed  the vision front end, three launches as mmr_encoder_forward_pixels makes them (H 768): pixels
 *       fp32 [B, C, image_size, image_size] -> patch16 bf16 [B * NP, C * patch^2] (the patch matrix: NP = (image_size /
 *       patch)^2 patches in row-major order, columns in (c, kh, kw) order, values bf16(pixel)) -> patch_out fp32 [B * NP, H]
 *       = patch16 . patch_w^T (patch_w bf16 [H, C * patch^2]) -> x fp32 [B * (NP + 1), H]: per image, row 0 = cls + pos[0],
 *       row 1 + p = patch_out[p] + pos[1 + p], each then LayerNorm(ln_g, ln_b, ln_eps).  patch16 and patch_out are written.
 */
int mmr_debug_enc_gemm(int32_t epi, int32_t nt, int32_t fold_ln, int32_t M, int32_t N, int32_t K, const void* x_dev,
                       const float* ln_src_dev, const float* ln_g_dev, const float* ln_b_dev, float ln_eps, float* ln_out_dev,
                       const void* w_dev, const float* bias_dev, const float* residual_dev, float* out_f32_dev,
                       void* out_bf16_dev, void* stream);
int mmr_debug_enc_attention(int32_t tensor_cores, int32_t B, int32_t S, int32_t H, int32_t heads, int32_t causal,
                            const float* qkv_dev, const int32_t* mask_dev, void* ctx_dev, void* stream);
int mmr_debug_enc_layernorm(int32_t H, int32_t M, const float* x_dev, const float* g_dev, const float* b_dev, float eps,
                            float* out_f32_dev, void* out_bf16_dev, void* stream);
int mmr_debug_enc_patch_embed(int32_t H, int32_t C, int32_t image_size, int32_t patch, int32_t B, const float* pixels_dev,
                              const void* patch_w_dev, const float* cls_dev, const float* pos_dev, const float* ln_g_dev,
                              const float* ln_b_dev, float ln_eps, void* patch16_dev, float* patch_out_dev, float* x_dev,
                              void* stream);

/* Introspection used by bench.py / tests: launches issued by this library since load, device facts. */
int64_t mmr_launch_count(void);
int mmr_device_sm_count(int device, int* out_sms);
/* Which kernel family the last mmr_search on this thread used: 1 = K1 stream, 2 = K2 umma, 3 = varlen. */
int mmr_last_kernel(void);
/* Queries the rescoring mode could not prove exact and reran on K1, since load. */
int64_t mmr_rescore_reruns(void);

#ifdef __cplusplus
}
#endif
#endif /* MMR_B200_H_ */
