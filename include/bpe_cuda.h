/*
 * bpe_cuda.h — C ABI of the B200 (sm_100a) BPE merge-loop engine.
 *
 * This is the drop-in boundary for the ONE hot path of neofytr/LLMTokenizer: the merge loop of
 * compress() (reference bpe/src/bpe.c:669-783: pair count -> most frequent pair -> rewrite of the
 * uint32 token stream).  Plain C types only; every output buffer is malloc()-owned so the caller
 * can hand it to free()/realloc() exactly as main.c:22 does with compress()'s encoding.
 *
 * What each entry point replaces in the reference (file:line relative to the reference tree):
 *   bpe_cuda_train            bpe/src/bpe.c:565-811  (widen, 16-thread get_freq + hash_table_merge,
 *                             collect + dyn_arr_max, rewrite, loop to exhaustion)
 *   bpe_cuda_encode           bpe/src/bpe.c:760-772 applied for a given merge list, ranks in id
 *                             order (the reference has no stand-alone encoder; additive)
 *   bpe_cuda_ctx_*            the same two operations split into upload / run / download so a
 *                             caller (bench, multi-process ranks) can keep the corpus resident in
 *                             HBM and shard it across GPUs; additive
 *   bpe_cuda_decode           bpe/src/bpe.c:341-394 decompress() with resolve_pair() bpe.c:23-92: ids ->
 *   bpe_cuda_ctx_decode*      bytes through the merge list; byte-exact and NUL-safe (explicit lengths
 *                             instead of the reference's NUL-terminated memo strings)
 *   bpe_cuda_encode_batch     encode / decode of a batch of independent documents in one call, with
 *   bpe_cuda_decode_batch     per-document offsets (the ids / bytes of document i are one slice of the
 *   bpe_cuda_ctx_*_batch      output); additive
 *   bpe_cuda_train_file       bpe/src/bpe.c:130-180 (get_file) + :555 (strlen cut) + :580-584 (widen) in front of the
 *   bpe_cuda_encode_file      path: the file is read in 32 MB pieces through pinned buffers, piece i+1 being read while
 *   bpe_cuda_ctx_upload_file  piece i is copied to the GPU and the pieces before it are widened and counted there
 *   bpe_cuda_free             free() of compress()'s outputs (main.c:22)
 *   bpe_cuda_last_error       perror/printf diagnostics of bpe.c:133-171,560
 *
 * Results are bit-identical to the reference: merge list, vocabulary and encoded ids, including
 * the reference's tie-break (first maximum in merged-hash-table iteration order, see DESIGN.md).
 *
 * There is no CPU fallback: every function fails with BPE_CUDA_ERR_CUDA when no sm_100 device or
 * driver is present.
 */
#ifndef BPE_CUDA_H
#define BPE_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* layout-identical to the reference's pair_t (bpe/inc/bpe.h:14-17) */
typedef struct
{
    uint32_t a, b;
} bpe_pair_t;

typedef struct
{
    uint64_t n_input;          /* tokens before the first merge (bytes up to the first NUL)        */
    uint64_t n_merges;         /* merges learned (train) / ranks in the table (encode)             */
    uint64_t n_tokens;         /* tokens after the last merge, summed over all ranks               */
    uint64_t ranks_applied;    /* encode: ranks whose pair occurred                                */
    uint64_t same_bucket_ties; /* iterations decided by chain order inside one hash bucket         */
    uint64_t threshold_edges;  /* iterations where D sat exactly on a table-doubling threshold     */
    uint64_t resolver_runs;    /* iterations resolved by the exact chain-order kernels             */
    uint64_t census_runs;      /* iterations that ran the 16-slice distinct-pair census            */
    uint64_t table_rehashes;
    uint64_t table_capacity;
    uint64_t final_distinct;   /* D when the loop stopped                                          */
    uint64_t kernel_launches;  /* kernels of this library launched by the call                     */
    uint64_t replace_launches; /* launches of the fused replace+scan+delta kernel                  */
    uint64_t replace_bytes;    /* algorithmic bytes of those launches: sum 4*(n_k + n_{k+1})       */
    double replace_ms;         /* their summed device time (only when profiling is enabled)        */
    double ms_device;          /* CUDA-event time of the whole run on this rank's stream           */
    double ms_h2d, ms_d2h;     /* host<->device copies (host-buffer entry points only)             */
    double ms_total;           /* wall clock of the call                                           */
    uint64_t worker_buckets[16]; /* emulated bucket counts of the reference's 16 worker tables      */
    /* only when profiling is enabled: device time of the other step kernels and of host-induced gaps */
    double select_ms, apply_ms, gap_ms;
    uint64_t replace_passes;   /* passes over the stream (a pass may carry several merges)            */
    uint64_t batch_merges;     /* merges that rode along in another merge's pass                       */
    uint64_t batch_passes;     /* passes that carried more than one merge                              */
} bpe_cuda_stats_t;

#define BPE_CUDA_OK 0
#define BPE_CUDA_ERR_ARG (-1)   /* NULL argument / invalid merge list                    */
#define BPE_CUDA_ERR_SHORT (-2) /* fewer than 2 characters (reference bpe.c:558-563)     */
#define BPE_CUDA_ERR_NOMEM (-3)
#define BPE_CUDA_ERR_CUDA (-4)  /* CUDA / NCCL failure, or no usable device              */
#define BPE_CUDA_ERR_STATE (-5) /* internal invariant broken (reported, never ignored)   */

/* ---- one-call entry points (host buffers in, malloc'd host buffers out) ------------------- */

/* Train on bytes[0..n) cut at the first 0x00 (bpe.c:555).  max_merges = 0 trains to exhaustion
 * like the reference (stop when the best frequency is <= 1, bpe.c:745, or no pair is left,
 * bpe.c:730).  n_gpus >= 1 shards the corpus over the first n_gpus devices of this process. */
int bpe_cuda_train(const uint8_t *bytes, size_t n, uint64_t max_merges, int n_gpus, bpe_pair_t **merges_out,
                   size_t *n_merges, uint32_t **tokens_out, size_t *n_tokens, bpe_cuda_stats_t *stats);

/* Apply merges[r] -> id 256+r for r = 0..n_merges-1, each as one greedy left-to-right pass. */
int bpe_cuda_encode(const uint8_t *bytes, size_t n, const bpe_pair_t *merges, size_t n_merges, int n_gpus,
                    uint32_t **tokens_out, size_t *n_tokens, bpe_cuda_stats_t *stats);

/* Inverse of encode: expand tokens[0..n_tokens) through the merge list (id 256+r -> merges[r]).
 * *bytes_out holds *n_bytes bytes plus one terminating 0 like decompress()'s string (bpe.c:390). */
int bpe_cuda_decode(const uint32_t *tokens, size_t n_tokens, const bpe_pair_t *merges, size_t n_merges, uint8_t **bytes_out,
                    size_t *n_bytes, bpe_cuda_stats_t *stats);

/* The same two operations on a FILE (what compress(path, ...) does, bpe.c:541-555): bytes after the first 0x00 are
 * ignored; n_gpus > 1 gives every rank its own byte range of the file to read. */
int bpe_cuda_train_file(const char *path, uint64_t max_merges, int n_gpus, bpe_pair_t **merges_out, size_t *n_merges,
                        uint32_t **tokens_out, size_t *n_tokens, bpe_cuda_stats_t *stats);
int bpe_cuda_encode_file(const char *path, const bpe_pair_t *merges, size_t n_merges, int n_gpus, uint32_t **tokens_out,
                         size_t *n_tokens, bpe_cuda_stats_t *stats);

/* Encode n_docs documents independently: document i is bytes[offsets[i] .. offsets[i+1]) (offsets: n_docs + 1
 * non-decreasing values), cut at its first 0x00.  ids of document i = tokens[tok_offsets[i] .. tok_offsets[i+1]),
 * identical to bpe_cuda_encode() of that document alone.  Device 0; outputs malloc()'d (tok_offsets: n_docs + 1).
 * One fixed sequence of kernel launches per batch, whatever the number of documents or merges.  Device memory: about
 * 10 B per input byte (BPE_CUDA_ERR_NOMEM beyond what is free).  A document must be shorter than 4 GiB.  Each document
 * is encoded by one thread block; one longer than a few hundred KB is slow this way (about 29 s for 4 MB with a
 * 32,000-merge table on a B200), and bpe_cuda_encode() is the faster path for it. */
int bpe_cuda_encode_batch(const uint8_t *bytes, const uint64_t *offsets, size_t n_docs, const bpe_pair_t *merges,
                          size_t n_merges, uint32_t **tokens_out, uint64_t **tok_offsets_out, size_t *n_tokens,
                          bpe_cuda_stats_t *stats);

/* Inverse of bpe_cuda_encode_batch: document i is tokens[tok_offsets[i] .. tok_offsets[i+1]) (tok_offsets: n_docs + 1
 * non-decreasing values; tok_offsets[0] need not be 0).  Its bytes are (*bytes_out)[byte_offsets[i] ..
 * byte_offsets[i+1]) (byte_offsets[0] = 0), identical to bpe_cuda_decode() of its ids alone, so the whole output is
 * bpe_cuda_decode() of tokens[tok_offsets[0] .. tok_offsets[n_docs]).  Device 0; outputs malloc()'d (*bytes_out with one
 * terminating 0 after *n_bytes bytes, *byte_offsets_out with n_docs + 1 values).  At most 4,294,967,294 documents.  An
 * id >= 256 + n_merges fails with BPE_CUDA_ERR_ARG, and bpe_cuda_last_error() names the first document that holds one.
 * One fixed sequence of four kernel launches whatever the number of documents (none when there is no id).  stats:
 * n_input = ids, n_tokens = bytes, n_merges, kernel_launches, ms_device (CUDA events around the kernels), ms_h2d,
 * ms_d2h, ms_total, and table_rehashes = 1 when the call flattened and uploaded the vocabulary. */
int bpe_cuda_decode_batch(const uint32_t *tokens, const uint64_t *tok_offsets, size_t n_docs, const bpe_pair_t *merges,
                          size_t n_merges, uint8_t **bytes_out, uint64_t **byte_offsets_out, size_t *n_bytes,
                          bpe_cuda_stats_t *stats);

void bpe_cuda_free(void *p);
const char *bpe_cuda_last_error(void);
int bpe_cuda_device_count(void);

/* ---- context API: one context per GPU (one per process rank, or several per process) ------ */
typedef struct bpe_cuda_ctx bpe_cuda_ctx_t;

int bpe_cuda_ctx_create(int device, bpe_cuda_ctx_t **ctx);
void bpe_cuda_ctx_destroy(bpe_cuda_ctx_t *ctx);

/* Multi-GPU: every rank calls this with the same 128-byte id obtained from
 * bpe_cuda_nccl_unique_id() on one rank (ship it with any bootstrap, e.g. torch.distributed). */
int bpe_cuda_nccl_unique_id(void *id128);
int bpe_cuda_ctx_set_comm(bpe_cuda_ctx_t *ctx, int rank, int world, const void *id128);

/* Copy this rank's contiguous shard of the (already NUL-cut) corpus into HBM.  The shard stays
 * resident; train/encode can be run on it repeatedly. */
int bpe_cuda_ctx_upload(bpe_cuda_ctx_t *ctx, const uint8_t *shard, size_t n_shard);
/* Fill the resident shard from a pointer that is already in device memory (no copy through the host). */
int bpe_cuda_ctx_upload_device(bpe_cuda_ctx_t *ctx, const void *dev_bytes, size_t n_shard);

/* Bytes [offset, offset + max_len) of a file become the resident shard, cut at the first 0x00 (*nul_found says whether
 * there was one: ranks that hold later parts of the file must then drop theirs, bpe_cuda_ctx_truncate(ctx, 0)).
 * Chunked, pinned, double-buffered; the shard is widened and its byte pairs counted while later chunks arrive. */
int bpe_cuda_ctx_upload_file(bpe_cuda_ctx_t *ctx, const char *path, uint64_t offset, uint64_t max_len, size_t *n_shard,
                             int *nul_found);
int bpe_cuda_ctx_truncate(bpe_cuda_ctx_t *ctx, size_t n_shard);

int bpe_cuda_ctx_train(bpe_cuda_ctx_t *ctx, uint64_t max_merges, bpe_cuda_stats_t *stats);
int bpe_cuda_ctx_encode(bpe_cuda_ctx_t *ctx, const bpe_pair_t *merges, size_t n_merges, bpe_cuda_stats_t *stats);

/* bpe_cuda_encode_batch() on a context, into caller buffers: tokens has room for offsets[n_docs] - offsets[0] ids
 * (ids <= bytes), tok_offsets for n_docs + 1 values.  Leaves the resident shard and the last train/encode results
 * untouched.  The pair -> rank table stays on the context and is rebuilt only when the merge list changes, so a
 * stream of batches with one vocabulary pays for it once. */
int bpe_cuda_ctx_encode_batch(bpe_cuda_ctx_t *ctx, const uint8_t *bytes, const uint64_t *offsets, size_t n_docs,
                              const bpe_pair_t *merges, size_t n_merges, uint32_t *tokens, uint64_t *tok_offsets,
                              bpe_cuda_stats_t *stats);

/* bpe_cuda_decode_batch() on a context: the n_docs + 1 byte offsets go to the caller's byte_offsets, *n_bytes is the
 * size of the output, and the bytes stay on the device like those of bpe_cuda_ctx_decode() (fetch them with
 * bpe_cuda_ctx_decode_download() or bpe_cuda_ctx_device_decoded()).  Leaves the resident shard and the last
 * train/encode results untouched.  The flattened vocabulary stays on the context and is rebuilt only when the merge list
 * changes (bpe_cuda_ctx_decode() shares it), so a stream of batches with one vocabulary pays for it once.  After an id
 * outside the vocabulary (BPE_CUDA_ERR_ARG) the context stays usable. */
int bpe_cuda_ctx_decode_batch(bpe_cuda_ctx_t *ctx, const uint32_t *tokens, const uint64_t *tok_offsets, size_t n_docs,
                              const bpe_pair_t *merges, size_t n_merges, uint64_t *byte_offsets, size_t *n_bytes,
                              bpe_cuda_stats_t *stats);

/* Results of the last train/encode on this context. */
int bpe_cuda_ctx_result_sizes(bpe_cuda_ctx_t *ctx, size_t *n_merges, size_t *n_tokens_local);
int bpe_cuda_ctx_download(bpe_cuda_ctx_t *ctx, bpe_pair_t *merges, uint32_t *tokens_local);
/* the same into pageable (malloc'd) memory: 32 MB pieces through two pinned staging buffers, the host copy of one piece
 * overlapping the DMA of the next */
int bpe_cuda_ctx_download_pageable(bpe_cuda_ctx_t *ctx, bpe_pair_t *merges, uint32_t *tokens_local);
/* device pointer to this rank's token stream after the last run (valid until the next run) */
const uint32_t *bpe_cuda_ctx_device_tokens(bpe_cuda_ctx_t *ctx);

/* Decode this rank's token stream of the last run without leaving the device; the bytes stay in HBM
 * (bpe_cuda_ctx_device_decoded) until the next decode.  _compare counts the bytes that differ from
 * the resident shard (UINT64_MAX when the lengths differ): the round trip decode(encode(x)) == x at
 * full scale with no host copy.  Shards decode independently: no collective.  (With several ranks a merged
 * token may straddle a shard boundary - it belongs to the left shard - so only the CONCATENATION of the ranks'
 * decodes equals the corpus; _compare is meant for a single rank.) */
int bpe_cuda_ctx_decode(bpe_cuda_ctx_t *ctx, const bpe_pair_t *merges, size_t n_merges, size_t *n_bytes);
int bpe_cuda_ctx_decode_download(bpe_cuda_ctx_t *ctx, uint8_t *bytes);
int bpe_cuda_ctx_decode_compare(bpe_cuda_ctx_t *ctx, uint64_t *n_diff);
const uint8_t *bpe_cuda_ctx_device_decoded(bpe_cuda_ctx_t *ctx);

/* knobs: "profile_replace" (0/1), "batch_steps" (merge steps enqueued per host poll),
 * "smem_hist_max_vocab", "batch_max" (merges per pass, 1 = off), "batch_min_z", "ranges",
 * "xchg_cap" (initial entries per inbox slot).  Returns 0 if the knob exists. */
int bpe_cuda_ctx_set_option(bpe_cuda_ctx_t *ctx, const char *name, long long value);

#ifdef __cplusplus
}
#endif
#endif /* BPE_CUDA_H */
