/* tokengeex_b200 — C ABI of the B200-native TokenGeeX hot path.
 *
 * Drop-in boundary for the data-parallel hot path of rojas-diego/tokengeex: UnigramLM
 * Viterbi segmentation (encode / encode_batch) and the forward-backward expected-count
 * pass + token-frequency pass that drive EM vocabulary pruning.  The reference is a
 * pure-Rust crate with no FFI of its own; these entry points are what a Rust `extern
 * "C"` shim inside the crate would bind (INTEGRATION.md shows that shim).  Each function
 * cites the reference interface it replaces (paths relative to the reference checkout).
 *
 * Conventions
 *  - plain pointers + sizes; no exceptions cross the boundary; every function returns a
 *    tgx_status (0 = ok) and tgx_last_error() describes the last failure on this thread.
 *  - "blob + offsets" layout for ragged data: item i occupies blob[off[i] .. off[i+1]),
 *    off has count+1 entries, off[0] == 0.
 *  - token ids are uint32 (TokenID = u32, src/lib.rs:19); id == index in the vocab array.
 *  - `_dev` variants take DEVICE pointers (text 16-byte aligned) and leave results in
 *    device memory; the others take HOST pointers and perform the H2D / D2H copies.
 *    Stream contract of the `_dev` variants: the library works on streams of its own.  Work queued on the legacy
 *    default stream (where torch and plain CUDA runtime calls put it unless told otherwise) before the call is ordered
 *    before the library's kernels; a caller that produces its buffers on another stream synchronises that stream
 *    first.  Results are complete when the call returns.
 *  - there is NO CPU fallback: without a CUDA device every compute entry point fails with
 *    TGX_ERR_NO_DEVICE.
 */
#ifndef TOKENGEEX_B200_H
#define TOKENGEEX_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct tgx_model tgx_model; /* opaque; replaces tokengeex::Model (src/model.rs:8-13) */

typedef enum tgx_status {
  TGX_OK = 0,
  TGX_ERR_INVALID = 1,     /* bad argument */
  TGX_ERR_UNSUPPORTED = 2, /* vocab beyond device limits (token > 64 B, >= 2^24 tokens/slots) */
  TGX_ERR_NO_DEVICE = 3,   /* no CUDA device / model created host-only */
  TGX_ERR_CUDA = 4,        /* CUDA runtime failure (message in tgx_last_error) */
  TGX_ERR_CAPACITY = 5,    /* output buffer too small; required size reported */
  TGX_ERR_NO_PATH = 6,     /* Error::NoPath(pos,len) (src/lib.rs:219-224,243-245) */
  TGX_ERR_BAD_Z = 7,       /* E-step: normalisation constant not "normal" (src/prune.rs:90-96) */
  TGX_ERR_NOT_UTF8 = 8     /* a corpus sample is not valid UTF-8 (load_sources, src/cli.rs:237-314) */
} tgx_status;

/* flags */
#define TGX_FLAG_CRLF 1u /* apply CrlfProcessor::preprocess (src/processor.rs:47-49) per sample */

typedef struct tgx_model_info {
  uint64_t vocab_size;
  uint32_t max_token_len;
  uint32_t trie_nodes;
  uint32_t trie_slots; /* 16-byte slots of the device double-array */
  uint32_t trie_terminals;
  int32_t device; /* -1 = host-only */
} tgx_model_info;

/* Last error message of the calling thread ("" if none). */
const char* tgx_last_error(void);

/* Model::from(vocab) (src/model.rs:16-30): builds the vocabulary trie — here an XOR
 * double-array — and uploads it to `device`.  Duplicate byte strings keep the LAST id
 * (src/trie.rs:19); the empty token never matches (src/trie.rs:51-63).
 * device >= 0: CUDA ordinal.  device == -1: host-only model (trie queries only). */
int tgx_model_create(const uint8_t* token_bytes, const uint64_t* token_offsets, const double* scores,
                     uint64_t vocab_size, int device, tgx_model** out);
/* `*model = Model::from(vocab)` as the EM loop does after every M-step / prune step (src/prune.rs:48,53), in
 * place: a new trie for the new vocabulary on the same device; streams and workspaces are kept (a fresh handle
 * would free and re-allocate GBs of scratch per EM sub-iteration).  When the new vocabulary is a subset of the one the
 * trie was built for (what the EM loop hands over) and not much smaller, the trie's layout is kept and only terminals,
 * ids and scores are rewritten (option 45; trie_slots of tgx_model_get_info then stays what it was): the same matches
 * as a fresh build.  On failure the model is unchanged.  Must not run concurrently with compute calls on the same
 * handle from other threads that still expect the old vocabulary. */
int tgx_model_rebuild(tgx_model* m, const uint8_t* token_bytes, const uint64_t* token_offsets, const double* scores,
                      uint64_t vocab_size);
void tgx_model_destroy(tgx_model* m);
int tgx_model_get_info(const tgx_model* m, tgx_model_info* info);

/* Model::common_prefix_search (src/model.rs:132-138 over src/trie.rs:22-63): ids and
 * lengths of every vocab token that prefixes text, ascending length.  Host-side walk of
 * the same double-array.  Writes min(count, cap) entries, returns the count in *count. */
int tgx_model_common_prefix_search(const tgx_model* m, const uint8_t* text, uint64_t n, uint32_t* ids,
                                   uint32_t* lens, uint64_t cap, uint64_t* count);

/* CrlfProcessor::preprocess over a batch (src/processor.rs:47-49; applied per sample as in
 * Tokenizer::encode_ordinary src/tokenizer.rs:92-99 and load_sources src/cli.rs:279-285).
 * out_text needs off[S] bytes; out_off S+1 entries. */
int tgx_crlf_batch(tgx_model* m, const uint8_t* text, const uint64_t* off, uint64_t S, uint8_t* out_text,
                   uint64_t* out_off);

/* Tokenizer::encode_ordinary_batch(inputs, dropout = 0.0) (src/tokenizer.rs:114-123) =
 * per sample: processors (crlf if TGX_FLAG_CRLF) then Model::encode (src/model.rs:59-129).
 *  ids      [ids_cap]  concatenated token ids, input order; ids_cap >= off[S] always suffices
 *  id_off   [S+1]      offsets into ids
 *  status   [S]        0 ok, TGX_ERR_NO_PATH for NoPath (may be NULL)
 *  proc_len [S]        length after the processors — the `len` of NoPath(len,len) (may be NULL)
 * Returns TGX_OK, or TGX_ERR_NO_PATH when any sample failed (*first_bad = lowest failing
 * index, as `collect::<Result<_>>` surfaces one error; other samples are still encoded),
 * or TGX_ERR_CAPACITY (id_off[S] holds the required capacity). */
int tgx_encode_batch(tgx_model* m, const uint8_t* text, const uint64_t* off, uint64_t S, uint32_t flags,
                     uint32_t* ids, uint64_t ids_cap, uint64_t* id_off, int32_t* status, uint64_t* proc_len,
                     int64_t* first_bad);
/* Same with device-resident inputs and outputs.  n_bytes = off[S].  *total_ids (host)
 * receives id_off[S].  d_off must be non-decreasing with samples shorter than 2^32 bytes (the host variants check it
 * and return TGX_ERR_INVALID / TGX_ERR_UNSUPPORTED; the device variants do not read the offsets on the host). */
int tgx_encode_batch_dev(tgx_model* m, const uint8_t* d_text, const uint64_t* d_off, uint64_t S,
                         uint64_t n_bytes, uint32_t flags, uint32_t* d_ids, uint64_t ids_cap,
                         uint64_t* d_id_off, int32_t* d_status, uint64_t* d_proc_len, uint64_t* total_ids,
                         int64_t* first_bad);

/* A corpus file image -> token ids: load_sources (src/cli.rs:237-314; samples separated by NUL bytes, docs/DATASET.md:69,
 * empty samples dropped, every sample strict UTF-8) followed by Model::encode of every sample (src/model.rs:59-129) —
 * the ordinary encoding: special tokens in the text are not split out.  The sample boundaries, the UTF-8 check and the
 * compaction run on the device (corpus_count / corpus_scatter), in chunks of ~option 7 bytes cut after a NUL byte
 * (a sample longer than a chunk enlarges it; samples must be shorter than 4 GiB).
 *  data[n]      the corpus image, host memory (pinned memory gives full speed)
 *  flags        TGX_FLAG_CRLF: CrlfProcessor per sample after the split ("\r" NUL "\n" stays two samples)
 *  sample_base  index of the buffer's first non-empty sample in the whole file: the dropout draw is keyed by
 *               sample_base + index (tgx_model_set_dropout), so ids do not depend on how a file is cut into buffers
 *  sep_id       -1 = none, else appended after every sample (the last one included)
 *  id_bytes     2 or 4: width of ids; with 2 the vocabulary and sep_id must be below 65536 (else TGX_ERR_UNSUPPORTED)
 *  ids          [ids_cap] of id_bytes each; ids_cap >= n + 1 always suffices
 *  id_off       [off_cap], n_samples + 1 entries written: sample i (its separator included) is ids[id_off[i] ..
 *               id_off[i+1]); off_cap >= (NUL bytes in data) + 2 always suffices
 *  n_samples / n_ids  non-empty samples and ids written (also when TGX_ERR_CAPACITY reports what is needed)
 * Returns TGX_OK; TGX_ERR_NOT_UTF8 (*first_bad = lowest invalid sample, relative to the buffer, *bad_pos = byte offset
 * of its first byte in data; nothing else is defined); TGX_ERR_NO_PATH (*first_bad = lowest failing sample, *bad_pos =
 * its length after processing; the other samples are encoded); TGX_ERR_CAPACITY.  The handle's dropout applies as for
 * tgx_encode_batch. */
int tgx_encode_corpus(tgx_model* m, const uint8_t* data, uint64_t n, uint32_t flags, uint64_t sample_base,
                      int64_t sep_id, uint32_t id_bytes, void* ids, uint64_t ids_cap, uint64_t* id_off,
                      uint64_t off_cap, uint64_t* n_samples, uint64_t* n_ids, int64_t* first_bad, uint64_t* bad_pos);

/* ModelVocabularyPruner::run_e_step (src/prune.rs:64-120): forward-backward expected
 * counts (Lattice::populate_marginal, src/lattice.rs:245-312, over Model::populate_nodes
 * src/model.rs:34-55) summed over all snippets of at most snippet_len bytes
 * (MAX_SAMPLE_LENGTH = 81920, src/prune.rs:75).  expected[V] is OVERWRITTEN with this
 * batch's sum (f64).  Returns TGX_ERR_BAD_Z if some snippet's z is not normal
 * (*bad_sample = lowest such sample, *bad_z its z); expected is then undefined. */
int tgx_expected_counts(tgx_model* m, const uint8_t* text, const uint64_t* off, uint64_t S,
                        uint64_t snippet_len, double* expected, int64_t* bad_sample, double* bad_z);
/* Device variant: d_expected[V] is ACCUMULATED into (+=) so a caller can sum shards /
 * chunks in place (and all-reduce the same buffer across GPUs). */
int tgx_expected_counts_dev(tgx_model* m, const uint8_t* d_text, const uint64_t* d_off, uint64_t S,
                            uint64_t n_bytes, uint64_t snippet_len, double* d_expected, int64_t* bad_sample,
                            double* bad_z);

/* The same E-step with the counts in exact integer form: limbs[5 * id + 0 .. 4] += (the four 32-bit words of the
 * 128-bit fraction, low to high, and the integer part) of token id's count.  The kernels accumulate in 192-bit fixed
 * point with integer atomics, so a count is the EXACT sum of its contributions (each truncated to 2^-128) —
 * bit-identical from run to run, for every chunking of the corpus and, after an integer (int64 SUM) all-reduce of the
 * limbs, for every number of GPUs — where the reference's f64 sum depends on rayon's completion order
 * (src/prune.rs:104-112).  Counts below ~1e-29 are below the resolution (the M-step's only threshold is 0.5).  A single
 * contribution must be below 2^64, the range of the integer word; only a lattice with positions nothing begins at
 * (beta = log 1 there, src/lattice.rs:275-287: vocabularies without every byte) can exceed it.
 * tgx_counts_from_limbs_dev turns (summed) limbs into the f64 vector the M-step reads: expected[id] = the exact sum
 * rounded to the nearest f64 (ties to even), overwritten.  tgx_expected_counts{,_dev} are this followed by that
 * conversion, so their f64 counts are the same correctly rounded values. */
int tgx_expected_counts_fixed_dev(tgx_model* m, const uint8_t* d_text, const uint64_t* d_off, uint64_t S,
                                  uint64_t n_bytes, uint64_t snippet_len, int64_t* d_limbs, int64_t* bad_sample,
                                  double* bad_z);
int tgx_counts_from_limbs_dev(tgx_model* m, const int64_t* d_limbs, uint64_t vocab_size, double* d_expected);

/* Frequency pass of prune_vocab (src/prune.rs:205-246): freq[id] += 1 over
 * Model::encode(sample, 0.0) of WHOLE samples.  freq[V] is overwritten (host variant) /
 * accumulated (device variant).  TGX_ERR_NO_PATH as for encode. */
int tgx_token_frequencies(tgx_model* m, const uint8_t* text, const uint64_t* off, uint64_t S, uint32_t flags,
                          uint64_t* freq, int64_t* first_bad, uint64_t* bad_len);
int tgx_token_frequencies_dev(tgx_model* m, const uint8_t* d_text, const uint64_t* d_off, uint64_t S,
                              uint64_t n_bytes, uint32_t flags, uint64_t* d_freq, int64_t* first_bad,
                              uint64_t* bad_len);

/* Pair-frequency pass of ModelVocabularyMerger::merge (src/merge.rs:36-84; SURVEY.md 8f rank 3): encode every
 * sample (dropout 0.0) and count the adjacent token-id pairs inside each sample.  pairs[i] = (first id << 32) |
 * second id and counts[i], for i < *n_pairs, ordered by count descending (`pairs.sort_unstable_by(|a, b|
 * b.1.cmp(&a.1))`, :83; equal counts — undefined order in the reference — by (first, second) ascending).
 * TGX_ERR_CAPACITY when there are more than cap distinct pairs (*n_pairs = needed); TGX_ERR_NO_PATH as for encode
 * (the reference unwraps the error, :59).  One call handles fewer than 2^31 tokens. */
int tgx_pair_frequencies(tgx_model* m, const uint8_t* text, const uint64_t* off, uint64_t S, uint32_t flags,
                         uint64_t* pairs, uint64_t* counts, uint64_t cap, uint64_t* n_pairs, int64_t* first_bad,
                         uint64_t* bad_len);
int tgx_pair_frequencies_dev(tgx_model* m, const uint8_t* d_text, const uint64_t* d_off, uint64_t S, uint64_t n_bytes,
                             uint32_t flags, uint64_t* d_pairs, uint64_t* d_counts, uint64_t cap, uint64_t* n_pairs,
                             int64_t* first_bad, uint64_t* bad_len);

/* ---- host half of the EM pruning loop (no device work; see tokengeex_b200/csrc/prune_host.cpp) ----
 * ModelVocabularyPruner::run_m_step (src/prune.rs:124-170, digamma :322-335).  kept[i] = 1 iff
 * token i survives (expected[i] >= 0.5 || keep[i]); new_scores[i] = digamma(max(expected[i],
 * 0.5)) - digamma(sum over survivors).  TGX_ERR_INVALID if a score is NaN/inf (reference panics). */
int tgx_m_step(const double* expected, const uint8_t* keep, uint64_t vocab_size, uint8_t* kept,
               double* new_scores, uint64_t* n_kept);
/* ModelVocabularyPruner::prune_vocab (src/prune.rs:173-319) given the token frequencies of its
 * frequency pass (tgx_token_frequencies): n-best alternatives per token (Lattice::nbest(2),
 * src/lattice.rs:152-238), loss ranking, cut at max(floor(V*shrink), target).  out_ids[*out_n] =
 * indices of the surviving tokens in their final (score-descending) order.  audit[8] optional. */
int tgx_prune_select(const uint8_t* token_bytes, const uint64_t* token_offsets, const double* scores,
                     const uint8_t* keep, uint64_t vocab_size, const uint64_t* freq, uint64_t n_samples,
                     uint64_t target_vocab_size, double shrink_factor, int threads, uint32_t* out_ids,
                     uint64_t* out_n, double* audit);

/* tgx_prune_select over the trie the model already holds: (token_bytes, token_offsets, scores) must be the vocabulary
 * of the last tgx_model_create / tgx_model_rebuild of `m` (checked by size only).  Saves the second trie build per
 * EM iteration (src/prune.rs:53 rebuilds the model right before prune_vocab walks it). */
int tgx_model_prune_select(tgx_model* m, const uint8_t* token_bytes, const uint64_t* token_offsets, const double* scores,
                           const uint8_t* keep, uint64_t vocab_size, const uint64_t* freq, uint64_t n_samples,
                           uint64_t target_vocab_size, double shrink_factor, int threads, uint32_t* out_ids,
                           uint64_t* out_n, double* audit);

/* Pinned host memory for callers that want asynchronous H2D/D2H (cudaHostAlloc). */
int tgx_host_alloc(void** p, uint64_t bytes);
int tgx_host_free(void* p);

/* Counters of the last compute call on this model (for bench.py): number of kernels
 * launched and device milliseconds of the dominant kernel(s), measured with CUDA events
 * on the model's stream.  what: 0 = kernels launched, 1 = Viterbi forward ms, 2 = fb-forward ms,
 * 3 = fb-backward ms, 4 = whole call device ms, 5 = backtrack ms, 6 = emit ms, 7 = match_kernel ms (forward passes over
 * the match stream; then 1 = the consumer of the stream alone: viterbi_rows_kernel / viterbi_team_kernel), 8 = the whole
 * forward pass (match + consumers + the wait for the side stream), 9 = the pair-CTA kernel of the longest samples on its
 * side stream (forward pass 3), 10 = the forward pass the call used (option 3; automatic resolves to 2 or 3), 11 = the
 * split kernels of tgx_encode_corpus summed over its chunks.  (For the chunked host entry points the others describe the
 * LAST chunk.) */
double tgx_model_last_stat(const tgx_model* m, int what);

/* Options.  Two of them are for callers:
 *    7 = bytes per chunk of the pipelined host entry points tgx_encode_batch / tgx_encode_corpus (default ~352 MiB);
 *   22 = byte offset of the E-step's text in the whole corpus when the call handles one shard of it (keyed dropout
 *        draw, see tgx_model_set_dropout).
 * The rest select between tested kernel variants and their launch shapes (bench / tests / tools/probe.py; not a stable
 * interface — defaults are what the measurements in profiles/ picked):
 *    3 = Viterbi forward pass when max_token_len <= 16: 4 = automatic (the default): 3 for a batch of at least 600 MiB,
 *        else 2; 2 = pair-CTA kernel; 3 = match stream + lane teams (tgx_team_kernel.cuh), the longest samples on the
 *        pair-CTA kernel beside them; 0 = match stream + row consumer (tgx_match_kernels.cuh); 1 = lane-group kernels
 *        (always used for longer tokens).  The forward pass 3 waits once, in the middle of the call, for the number of
 *        long samples (it sizes the grids);
 *   32 / 33 / 35 = forward pass 3: byte length from which a sample runs on the pair-CTA kernel (default 65536);
 *        match_kernel CTAs (slices of the blob) per SM; bytes of leading match rows staged in shared memory;
 *   45 = tgx_model_rebuild keeps the double-array's layout when the new vocabulary is a subset of the one it was built
 *        for and has at least this many per mille of its tokens (default 450; 0 = always build afresh);
 *   37 / 38 / 39 / 43 = match2_kernel (walks compacted inside their warp; 0 = match_kernel); long samples per pair CTA
 *        on the side stream of forward pass 3 (default 20); match2_kernel skips the positions inside those samples;
 *        groups per CTA of that side kernel (default 4);
 *   23 / 24 = match_kernel: threads per CTA, bytes of leading trie slots staged in shared memory;
 *   25 / 26 = viterbi_rows_kernel: warps per CTA, bytes of leading match rows staged in shared memory;
 *    0 / 1 = lane-group kernels: lanes per short sample (1,2,4,8,16,32), byte threshold from which a sample gets a
 *        full warp (also: warp-cooperative backtrack);
 *    6 / 13 / 14 = pair-CTA kernel: groups per CTA (0 = as many as fit), trie
 *        levels staged in shared memory (0..2), shape (0 = by batch size, 1 = 5 groups, 2 = 6 groups);
 *   11 = chunked host entry point queues the next chunk's kernels before the current chunk has finished (default 0);
 *   16 = emit looks token ids up in the token hash (1, default when max_token_len <= 16) or re-walks the trie (0);
 *    2 / 5 / 17 / 18 / 19 / 20 / 21 / 30 / 31 = E-step: lanes per snippet of the lane-group kernels; byte threshold from
 *        which a snippet gets a full warp (0 = automatic); byte threshold below which a snippet runs on ONE lane (< 0 =
 *        automatic, 0 = never); resident blocks per SM of the lane kernels; form (1, the default: beta chains stored and
 *        run beside the alpha chains, lane kernels that walk the trie, with or without the dropout draw;
 *        2: the lane kernels over the match stream always; 0: no beta array, lane-group kernels only); replicas
 *        (default 64) of the accumulators of the hottest ids (default: ids below 4096); per mille of the lane
 *        snippets, longest first, at which the first / second group of lane snippets ends (groups run on streams of
 *        their own: the counts of one beside the chains of the next). */
int tgx_model_set_option(tgx_model* m, int key, int64_t value);

/* The `dropout` argument of Model::encode (src/model.rs:59,100) for the encode entry points
 * (tgx_encode_batch{,_dev}) and of Model::populate_nodes (src/model.rs:34-55, called by run_e_step with the
 * pruner's dropout, src/prune.rs:87) for tgx_expected_counts{,_dev}; the frequency passes always encode with
 * dropout 0.0, as the reference does (src/prune.rs:218, src/merge.rs:58).  dropout must be in [0, 1); 0.0 (the default, and every
 * benchmark configuration) switches it off.  dropout >= 1.0 is not a draw at all — every multi-byte
 * token is skipped (src/model.rs:218-236) — and is served by a model created from the single-byte
 * tokens (see tokengeex_b200/tokenizer.py).
 * The reference draws rand::random::<f64>() from an unseeded thread_rng for every multi-byte candidate
 * of a reachable position, so only the distribution of its output is defined.  Here the draw of
 * candidate (sample index within the call, start byte within the processed sample, token length) is a
 * pure function of `seed` (two rounds of the splitmix64 finaliser, 53-bit uniform in [0, 1); the
 * candidate is kept iff dropout < u): independent uniform draws like the reference's, but
 * reproducible, independent of chunking and sharding, and restated in oracle/ for bit-exact tests.
 * In the E-step the candidate is (byte offset of its first byte in the call's text + option 22, token length):
 * option 22 of tgx_model_set_option = offset of the call's text in the whole corpus when it is one shard of it, so
 * that the lattices do not depend on the sharding; use a new seed for every E-step.
 * The setting belongs to the model handle and applies to the calls that follow it: threads that encode through one
 * handle with different dropout values serialise set + call themselves (tokengeex_b200/tokenizer.py holds a lock).
 * With dropout > 0 the forward pass runs on the pair kernel with the draw in its producers
 * (viterbi_pair_drop_kernel; lane-group viterbi_kernel<G, true> for tokens > 16 bytes) and the E-step on the lane kernels
 * over the match stream (fbr_split_kernel<true> / fbr_contrib_kernel<true>; lane-group kernels for tokens > 16 bytes). */
int tgx_model_set_dropout(tgx_model* m, double dropout, uint64_t seed);

#ifdef __cplusplus
}
#endif
#endif
