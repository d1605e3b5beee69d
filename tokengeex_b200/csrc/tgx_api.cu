// C ABI of the B200-native TokenGeeX hot path (include/tokengeex_b200.h) and the helper
// kernels around the Viterbi / forward-backward kernels of tgx_kernels.cuh.
//
// Compile: nvcc -gencode arch=compute_100a,code=sm_100a --fmad=false -lineinfo
// (--fmad=false: every f64 sum on the score path must round exactly like the
// reference's separate add instructions.)
#include <cub/cub.cuh>
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/tokengeex_b200.h"
#include "tgx_kernels.cuh"
#include "tgx_match_kernels.cuh"
#include "tgx_team_kernel.cuh"
#include "tgx_fb_rows_kernels.cuh"
#include "trie_build.h"

namespace {

thread_local std::string g_err;
int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}
#define CU(call)                                                                                   \
  do {                                                                                             \
    cudaError_t _e = (call);                                                                       \
    if (_e != cudaSuccess)                                                                         \
      return fail(TGX_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(_e));               \
  } while (0)

// Growable device buffer (never shrinks; reused across calls).
struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  cudaError_t reserve(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaMalloc(&p, want);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  template <class T>
  T* as() const { return reinterpret_cast<T*>(p); }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
};

struct Stats {
  double launches = 0, viterbi_ms = 0, fwd_ms = 0, bwd_ms = 0, total_ms = 0, back_ms = 0, emit_ms = 0, match_ms = 0,
         side_ms = 0, forward_ms = 0, algo = 0, split_ms = 0;
};

}  // namespace

// Scratch of one batch in flight: its compute stream, the stream its control words are read through, events and
// every intermediate buffer.  The model owns two, so that the chunked host entry point can have the kernels of
// chunk k+1 queued behind chunk k (the tail of a chunk is a handful of long samples on a few SMs).
struct Workspace {
  cudaStream_t stream = nullptr;
  // The compute stream never issues a D2H copy itself: measured on B200 (profiles/r01_ubench_overlap.txt),
  // once a stream has used the D2H copy engine its next kernels queue behind whatever that engine is
  // doing — here the bulk D2H of the previous chunk.  Control words are read through this stream.
  cudaStream_t stream_ctl = nullptr;
  cudaEvent_t ev_ctl = nullptr;
  // algo 3: the pair-CTA kernel of the batch's longest samples runs here, beside match + teams on `stream`
  cudaStream_t stream_side = nullptr;
  cudaStream_t stream_low = nullptr;  // lowest priority: the team CTAs that take over the SMs the pair-CTA kernel frees
  cudaEvent_t ev_side_fork = nullptr, ev_side_join = nullptr, ev_low_join = nullptr;
  int algo_used = 2;       // forward algorithm of the call in flight (tgx_model_last_stat 10)
  bool side_used = false;  // ev[10..11] were recorded by the call in flight
  unsigned long long* h_words = nullptr;  // pinned, 8 words
  cudaEvent_t ev[14] = {};  // [10..11] pair-CTA kernel on the side stream, [12] forward pass complete (algo 3)
  Stats stats;
  DevBuf text2, off2, bitmap, blk, ustart, ulen, keys_out, vals_in, vals_out, cubtmp, bp, mark, tilecnt, ntok, status,
      small, rec, skip;
};

struct tgx_model {
  tgx::DoubleArray da;
  uint64_t V = 0;
  uint64_t V_built = 0;        // vocabulary size the double-array's layout was built for
  int retarget_permille = 450; // tgx_model_rebuild keeps the layout for a subset of at least this share of V_built (0 = never)
  int device = -1;
  uint4* d_trie = nullptr;
  size_t trie_cap = 0;  // slots allocated at d_trie
  // emit: token hash (bytes -> id, one probe per token); hash.mask == 0 = not available
  tgx::TokenHash hash;
  DevBuf d_hash;
  // match tables (trie_build.h: slots8 / rows / row_ids; max_token_len <= 16 only): have_rows == false = not available
  DevBuf d_trie8, d_rows, d_rowids, d_pair2;
  bool have_rows = false;
  uint32_t rows16 = 0;  // 16-byte units in the row table
  Workspace ws[2];
  int wi = 0;  // workspace the next launches go to
  Workspace& w() { return ws[wi]; }
  const Workspace& w() const { return ws[wi]; }
  Stats last_stats;  // of the last finished call (tgx_model_last_stat)
  cudaStream_t stream2 = nullptr;  // long units run beside the short ones (E-step)
  cudaStream_t stream3 = nullptr;  // lane-per-snippet kernels (E-step)
  cudaStream_t stream4 = nullptr;  // beta chains of the warp-per-snippet kernels in split form
  cudaStream_t stream5 = nullptr, stream6 = nullptr;  // second / third group of lane snippets (E-step)
  cudaEvent_t ev_grp[4] = {}, ev_join5 = nullptr, ev_join6 = nullptr;
  int estep_cut1 = 150, estep_cut2 = 1000;  // per mille of the lane snippets (longest first) where the groups end
  cudaEvent_t ev_join3 = nullptr, ev_join4 = nullptr;
  cudaStream_t stream_h2d = nullptr, stream_d2h = nullptr;  // copy engines of the chunked host entry points
  cudaEvent_t ev_h2d[2] = {}, ev_d2h[2] = {};
  uint64_t* h_off = nullptr;       // pinned staging for rebased chunk offsets
  uint64_t h_off_cap = 0;
  unsigned char* h_out = nullptr;  // pinned staging for the small per-sample outputs (id_off, status, proc_len)
  uint64_t h_out_cap = 0;
  uint64_t chunk_bytes = 352ull << 20;  // ~3 chunks per GB: below that the longest sample's dp chain dominates a chunk
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev_caller = nullptr;
  std::recursive_mutex mu;
  // options
  int g_short = 8;
  int64_t long_threshold = 512;  // samples at least this long: full warp (lane-group forward kernels, backtrack)
  int g_estep = 4;
  // Snippets at least this long get a full warp (G = 32) on a second stream.  0 = automatic: a G-lane group runs a
  // position in ~8 us, so the longest snippet handed to the lane groups should not outlast the batch itself
  // (~3 GB/s): threshold = max(8192, n_bytes / 18000) — beyond 1.5 GB no snippet (<= 81920 B) takes the warp path
  // (tools/probe.py --what estep at 0.2, 0.6, 2 and 4 GB: best thresholds 16 K, 32 K, >= 64 K, none)
  int64_t estep_long_threshold = 0;
  // Snippets shorter than this run one LANE each (fb_*_lane_kernel; max_token_len <= 16).  0 = off, < 0 = automatic:
  // everything below the long threshold, and the automatic long threshold becomes 16000 + n_bytes / 30000 — measured on
  // B200 (tools/probe.py --what estep): lanes fold 8 GB/s of short snippets against 2.9 GB/s for 4-lane groups, but a
  // chain advances one position per ~4.3 us (forward) on a lane and per ~1.3 us on a warp, so the longest lane snippet
  // must not outlast the rest (best thresholds in split form: 24-32 K at 0.5 GB, 32-48 K at 1 GB, none — every snippet on a lane — at 4 GB).
  int64_t estep_lane_threshold = -1;
  // Lane kernels in split form: the backward chain only stores beta and runs beside the forward chain, a third
  // kernel adds the expected counts (needs 8 more bytes per input byte; falls back to the fused form without them).
  int estep_split = 1;
  int estep_rows = 1;  // E-step over the match stream (tgx_fb_rows_kernels.cuh) when the match tables exist
  // E-step: replicas of the count vector for the hot_k hottest (smallest) ids.  (4 GB / 500k tokens, tools/probe.py: 636 ms
  // with 32-128 replicas of 1024-4096 ids, 647 with 256 x 4096, 669 with 512 x 4096, 639 with 16 x 2048.)
  int hot_k = 4096, hot_r = 64;
  int lane_blocks_per_sm = 0;  // lane E-step kernels: resident 128-thread blocks per SM (0 = as many as fit, 9)
  // Viterbi forward (max_token_len <= 16; longer vocabularies always use the lane-group kernels):
  // 0 = match stream + row consumer (tgx_match_kernels.cuh), 1 = lane-group kernels, 2 = pair-CTA kernel (the default
  // of the first round; still what encodes with dropout in (0, 1)), 3 = match stream + lane teams with the longest
  // samples on the pair-CTA kernel beside them (tgx_team_kernel.cuh), 4 = automatic (the default): 3 for a batch of at
  // least `wide_bytes` bytes, else 2 — below that a batch is bound by its longest sample's chain, which the pair-CTA
  // kernel runs fastest (measured on B200: 1 GB 29.5 against 32.3 ms, 352 MB chunks 18 against 13.5 ms).
  int algo = 4;
  int match_threads = 1024;       // threads per CTA of match_kernel (one CTA per SM)
  int match_skip = 1;             // forward pass 3: no walks inside the samples the pair-CTA kernel takes
  int match_compact = 1;          // match2_kernel (walks compacted inside their warp) instead of match_kernel
  int match_ctas_per_sm = 8;      // match_kernel: CTAs (contiguous slices of the blob) per SM, handed out as SMs come free
  // algo 3: samples at least this long run on the pair-CTA kernel (16 lanes per sample: the shortest chain per
  // position) on a stream of its own, the rest four lanes each on viterbi_team_kernel over the match stream
  int64_t team_long_threshold = 65536;
  int side_groups = 4;   // ... and groups per CTA of that kernel: four (8 chains) run a chain in ~90 cycles per position, five in ~100
  int side_load = 20;    // algo 3: long samples per pair CTA on the side stream (10 chains each)
  int64_t team_hot_bytes = 160 << 10;  // leading bytes of the row table viterbi_team_kernel stages in shared memory
  int64_t match_stage_bytes = 64 << 10;  // leading trie slots (8 bytes each) match_kernel stages in shared memory
  int rows_warps = 16;            // warps per CTA of viterbi_rows_kernel (one CTA per SM; two samples per warp)
  int64_t rows_hot_bytes = 96 << 10;  // leading bytes of the row table viterbi_rows_kernel stages in shared memory
  int num_sms = 148;
  int groups = 0;       // consumer/producer groups per CTA of the pair kernel; 0 = as many as fit
  uint32_t pair_grid_cap = 0;  // CTAs the next pair-kernel launch may use (0 = one per SM); set and cleared by algo 3
  int smem_optin = 232448;
  // Chunked host entry point: queue chunk k+1's kernels (second workspace) before chunk k has finished.  Off by
  // default: measured on B200 (tools/e2e_trace.py, 1 GB) it LOSES, 75.4 vs 67.6 ms with two chunks — the next
  // chunk's persistent forward CTAs take every SM the moment the current forward kernel drains, and the current
  // chunk's backtrack / emit kernels then wait for registers until those CTAs exit.
  int overlap_chunks = 0;
  int hot_levels = 2;  // leading trie levels the pair kernel may stage in shared memory (0..2)
  int emit_hash = 1;   // emit: token ids through the token hash (1 probe per token) instead of re-walking the trie
  int pair_shape = 0;  // 0 = by batch size, 1 = latency shape (5 groups), 2 = throughput shape (6 groups)
  // tgx_model_set_dropout: Model::encode's dropout argument for the encode entry points (src/model.rs:59,100).
  // 0.0 = off (every BASELINE configuration); in (0, 1) the keyed draw of tgx_kernels.cuh::drop_draw.
  double dropout = 0.0;
  uint64_t drop_seed = 0;
  uint64_t drop_unit_base = 0;  // first sample of the chunk being queued (chunked host entry point)
  uint64_t drop_byte_base = 0;  // E-step: offset of this call's text in the whole (sharded) corpus, option 22
  uint64_t wide_bytes = 600ull << 20;
  // buffers of the host entry points (two sets for the chunk pipeline) and of the E-step / frequency pass
  DevBuf Bbeta, accfix;
  DevBuf text, off, idoff, A, expected, freq, ids, scount, hot, text_b, off_b, ids_b, idoff_b, scount_b;
  // tgx_encode_corpus, per buffer set: raw chunk, split scratch (tile counts and their scan, control words), the ids
  // as they leave the device (corpus_finalize); events around the split kernels (tgx_model_last_stat 11)
  DevBuf raw[2], split[2], fin[2];
  cudaEvent_t ev_split[2][4] = {};
};

// =========================================================================================
// helper kernels
// =========================================================================================
namespace tgxk {

constexpr int CRLF_BLOCK = 256;               // threads
constexpr int CRLF_PER_THREAD = 16;           // bytes
constexpr int CRLF_TILE = CRLF_BLOCK * CRLF_PER_THREAD;

// K1a: one bit per byte position that starts a sample (so "\r" | "\n" across a sample
// boundary is not merged: the processor runs per sample, src/tokenizer.rs:92-99).
__global__ void crlf_mark_starts(const uint64_t* __restrict__ off, uint64_t S, uint32_t* __restrict__ bitmap) {
  uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s == 0 || s >= S) return;
  uint64_t p = off[s];
  atomicOr(bitmap + (p >> 5), 1u << (p & 31));
}

// removed(p): text[p] == '\r' followed, inside the same sample, by '\n'
// (str::replace("\r\n", "\n"), src/processor.rs:47-49: left-to-right, non-overlapping —
// "\r\n" occurrences never overlap each other, so the predicate is position-local).
// One thread looks at 16 bytes (one aligned 16-byte load when the blob allows it) plus the byte
// after them.  Returns the 16-bit mask of removed bytes; `starts` receives the sample-start
// flags of positions base .. base+15; `nvalid` the number of bytes below N.
__device__ __forceinline__ uint32_t crlf_mask16(const uint8_t* __restrict__ text, uint64_t N,
                                                const uint32_t* __restrict__ bitmap, uint64_t base, uint4& v,
                                                uint32_t& starts, uint32_t& nvalid) {
  if (base >= N) {
    v = make_uint4(0, 0, 0, 0);
    starts = 0;
    nvalid = 0;
    return 0;
  }
  nvalid = (uint32_t)min((uint64_t)16, N - base);
  uint32_t next = 0;
  if (nvalid == 16) {
    v = *reinterpret_cast<const uint4*>(text + base);
    if (base + 16 < N) next = text[base + 16];
  } else {
    uint32_t w[4] = {0, 0, 0, 0};
    for (uint32_t i = 0; i < nvalid; i++) w[i >> 2] |= (uint32_t)text[base + i] << (8 * (i & 3));
    v = make_uint4(w[0], w[1], w[2], w[3]);
  }
  // start flags of positions base .. base+16 (bit i <-> position base + i)
  const uint32_t wi = (uint32_t)(base >> 5);
  const unsigned long long bits = (unsigned long long)bitmap[wi] | ((unsigned long long)bitmap[wi + 1] << 32);
  const uint32_t sb = (uint32_t)(bits >> (base & 31)) & 0x1FFFFu;
  starts = sb & 0xFFFFu;
  const uint32_t wv[4] = {v.x, v.y, v.z, v.w};
  uint32_t cr = 0, lf = 0;
#pragma unroll
  for (int i = 0; i < 16; i++) {
    const uint32_t c = (wv[i >> 2] >> (8 * (i & 3))) & 0xFFu;
    cr |= (uint32_t)(c == '\r') << i;
    lf |= (uint32_t)(c == '\n') << i;
  }
  lf |= (uint32_t)(next == '\n') << 16;
  // byte i is removed iff it is '\r', byte i+1 exists, is '\n' and does not start a sample
  uint32_t m = cr & (lf >> 1) & ~(sb >> 1);
  if (nvalid < 16) m &= (1u << nvalid) - 1u;  // the byte after the last valid one does not exist (next == 0)
  return m & 0xFFFFu;
}

__device__ __forceinline__ uint32_t block_exclusive_scan(uint32_t v, uint32_t* warp_sums, uint32_t* total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t x = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    uint32_t y = __shfl_up_sync(0xFFFFFFFFu, x, o);
    if (lane >= o) x += y;
  }
  if (lane == 31) warp_sums[warp] = x;
  __syncthreads();
  uint32_t before = 0, tot = 0;
#pragma unroll
  for (int i = 0; i < CRLF_BLOCK / 32; i++) {
    const uint32_t ws = warp_sums[i];
    if (i < warp) before += ws;
    tot += ws;
  }
  if (total) *total = tot;
  return before + x - v;
}

// K1b: removed bytes per 4096-byte tile.
__global__ void __launch_bounds__(CRLF_BLOCK) crlf_count(const uint8_t* __restrict__ text, uint64_t N,
                                                         const uint32_t* __restrict__ bitmap,
                                                         unsigned long long* __restrict__ blk_removed) {
  __shared__ uint32_t ws[CRLF_BLOCK / 32];
  const uint64_t base = (uint64_t)blockIdx.x * CRLF_TILE + (uint64_t)threadIdx.x * CRLF_PER_THREAD;
  uint4 v;
  uint32_t starts, nvalid;
  uint32_t c = __popc(crlf_mask16(text, N, bitmap, base, v, starts, nvalid));
#pragma unroll
  for (int o = 16; o; o >>= 1) c += __shfl_xor_sync(0xFFFFFFFFu, c, o);
  if ((threadIdx.x & 31) == 0) ws[threadIdx.x >> 5] = c;
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t t = 0;
#pragma unroll
    for (int i = 0; i < CRLF_BLOCK / 32; i++) t += ws[i];
    blk_removed[blockIdx.x] = t;
  }
}

// first index s in [0, S] with off[s] >= p
__device__ __forceinline__ uint64_t lower_bound_off(const uint64_t* __restrict__ off, uint64_t S, uint64_t p) {
  uint64_t lo = 0, hi = S + 1;
  while (lo < hi) {
    const uint64_t mid = (lo + hi) >> 1;
    if (off[mid] < p) lo = mid + 1; else hi = mid;
  }
  return lo;
}

// Compaction of one tile (CRLF_TILE bytes at most) through shared memory: the thread's 16 bytes `v` minus the bytes flagged
// in `m` go to stage[o ..], then the tile's `total` kept bytes are written to out[ob ..] with aligned 16-byte stores.
__device__ __forceinline__ void tile_compact_store(const uint4& v, uint32_t m, uint32_t nvalid, uint32_t o, uint64_t ob,
                                                   uint32_t total, uint8_t* stage, uint8_t* __restrict__ out) {
  const uint32_t wv[4] = {v.x, v.y, v.z, v.w};
  if (m == 0 && nvalid == 16 && (o & 3u) == 0) {
#pragma unroll
    for (int j = 0; j < 4; j++) *reinterpret_cast<uint32_t*>(stage + o + 4 * j) = wv[j];
  } else {
    uint32_t q = o;
#pragma unroll
    for (int i = 0; i < 16; i++)
      if (i < (int)nvalid && !((m >> i) & 1u)) stage[q++] = (uint8_t)(wv[i >> 2] >> (8 * (i & 3)));
  }
  __syncthreads();
  // ---- [ob, ob + total) of `out`: unaligned head and tail by bytes, the rest by 16-byte vectors
  const uint64_t oe = ob + total;
  const uint64_t a0 = min((uint64_t)((ob + 15) & ~15ull), oe);
  const uint32_t head = (uint32_t)(a0 - ob);
  if (threadIdx.x < head) out[ob + threadIdx.x] = stage[threadIdx.x];
  const uint32_t nvec = (uint32_t)((oe - a0) >> 4);
  for (uint32_t c = threadIdx.x; c < nvec; c += CRLF_BLOCK) {
    const uint32_t so = head + 16 * c;  // source offset in stage (any alignment)
    const uint32_t* sw = reinterpret_cast<const uint32_t*>(stage + (so & ~3u));
    const uint32_t sh = 8 * (so & 3u);
    uint32_t w[5];
#pragma unroll
    for (int j = 0; j < 5; j++) w[j] = sw[j];
    uint4 r;
    r.x = __funnelshift_r(w[0], w[1], sh);
    r.y = __funnelshift_r(w[1], w[2], sh);
    r.z = __funnelshift_r(w[2], w[3], sh);
    r.w = __funnelshift_r(w[3], w[4], sh);
    *reinterpret_cast<uint4*>(out + a0 + 16ull * c) = r;
  }
  const uint64_t t0 = a0 + 16ull * nvec;
  if (threadIdx.x < (uint32_t)(oe - t0)) out[t0 + threadIdx.x] = stage[(uint32_t)(t0 - ob) + threadIdx.x];
}

// K1c: compact every tile through shared memory and write it with aligned 16-byte stores; the
// thread that sees a sample start also writes that sample's new offset (found by binary search).
// blk_prefix = exclusive scan of blk_removed (n_tiles + 1 entries).
__global__ void __launch_bounds__(CRLF_BLOCK) crlf_scatter(const uint8_t* __restrict__ text, uint64_t N,
                                                           const uint64_t* __restrict__ off, uint64_t S,
                                                           const uint32_t* __restrict__ bitmap,
                                                           const unsigned long long* __restrict__ blk_prefix,
                                                           uint64_t n_tiles, uint8_t* __restrict__ out,
                                                           uint64_t* __restrict__ new_off) {
  __shared__ uint32_t ws[CRLF_BLOCK / 32];
  __shared__ __align__(16) uint8_t stage[CRLF_TILE + 32];
  const uint64_t tile_base = (uint64_t)blockIdx.x * CRLF_TILE;
  const uint64_t base = tile_base + (uint64_t)threadIdx.x * CRLF_PER_THREAD;
  uint4 v;
  uint32_t starts, nvalid;
  const uint32_t m = crlf_mask16(text, N, bitmap, base, v, starts, nvalid);
  const uint32_t kept = nvalid - __popc(m);
  uint32_t total;
  const uint32_t o = block_exclusive_scan(kept, ws, &total);
  const uint64_t ob = tile_base - blk_prefix[blockIdx.x];  // blob index (in `out`) of the tile's first kept byte
  // ---- new offsets of the samples that start inside this thread's 16 bytes
  uint32_t sb = starts;
  if (base == 0) sb |= 1u;  // position 0 starts sample 0 (and every empty sample before the first byte)
  if (nvalid < 16) sb &= (1u << nvalid) - 1u;
  while (sb) {
    const int i = __ffs(sb) - 1;
    sb &= sb - 1;
    const uint64_t p = base + i;
    const uint64_t np = ob + o + __popc(~m & ((1u << i) - 1u));
    for (uint64_t s = lower_bound_off(off, S, p); s <= S && off[s] == p; s++) new_off[s] = np;
  }
  if (blockIdx.x == n_tiles - 1 && threadIdx.x == 0) {  // samples that start at N (off[S], trailing empties)
    const uint64_t np = N - blk_prefix[n_tiles];
    for (uint64_t s = lower_bound_off(off, S, N); s <= S; s++) new_off[s] = np;
  }
  tile_compact_store(v, m, nvalid, o, ob, total, stage, out);
}

// ---- corpus split (tgx_encode_corpus): a raw chunk of NUL-separated samples -> blob + offsets of the non-empty
// samples, every sample checked to be strict UTF-8 (Unicode Table 3-7, what str::from_utf8 and Python's strict decode
// accept).  Same shape as the crlf kernels: per-thread 16-byte masks, counts per 4096-byte tile, one scan, scatter.

// Masks of the 16 positions base .. base+15 (bit i <-> base + i): `keep` = not NUL, `start` = first byte of a
// non-empty sample (a byte before position 0 counts as NUL), `bad` = where strict decoding fails.  Bytes at or beyond N
// read as NUL, so a sequence cut off by a NUL or by the end of the buffer fails at its lead byte.
__device__ __forceinline__ void corpus_mask16(const uint8_t* __restrict__ text, uint64_t N, uint64_t base, uint4& v,
                                              uint32_t& keep, uint32_t& start, uint32_t& bad, uint32_t& nvalid) {
  nvalid = base < N ? (uint32_t)min((uint64_t)16, N - base) : 0u;
  if (nvalid == 16) {
    v = *reinterpret_cast<const uint4*>(text + base);
  } else {
    uint32_t w[4] = {0, 0, 0, 0};
    for (uint32_t i = 0; i < nvalid; i++) w[i >> 2] |= (uint32_t)text[base + i] << (8 * (i & 3));
    v = make_uint4(w[0], w[1], w[2], w[3]);
  }
  // bit e <-> position base + e - 3: the three bytes before the thread's 16 and the three after them
  const uint32_t wv[4] = {v.x, v.y, v.z, v.w};
  uint32_t nul = 0, cont = 0, ge2 = 0, ge3 = 0, l4 = 0, badlead = 0, e0 = 0, ed = 0, f0 = 0, f4 = 0, c8 = 0, c9 = 0,
           ca = 0;
#pragma unroll
  for (int e = 0; e < 22; e++) {
    uint32_t c;
    if (e < 3) {
      c = (base + e >= 3 && base + e - 3 < N) ? text[base + e - 3] : 0u;
    } else if (e < 19) {
      c = (wv[(e - 3) >> 2] >> (8 * ((e - 3) & 3))) & 0xFFu;
    } else {
      c = base + e - 3 < N ? text[base + e - 3] : 0u;
    }
    nul |= (uint32_t)(c == 0) << e;
    cont |= (uint32_t)((c & 0xC0u) == 0x80u) << e;
    ge2 |= (uint32_t)(c >= 0xC2u && c <= 0xF4u) << e;
    ge3 |= (uint32_t)(c >= 0xE0u && c <= 0xF4u) << e;
    l4 |= (uint32_t)(c >= 0xF0u && c <= 0xF4u) << e;
    badlead |= (uint32_t)(c == 0xC0u || c == 0xC1u || c >= 0xF5u) << e;
    e0 |= (uint32_t)(c == 0xE0u) << e;
    ed |= (uint32_t)(c == 0xEDu) << e;
    f0 |= (uint32_t)(c == 0xF0u) << e;
    f4 |= (uint32_t)(c == 0xF4u) << e;
    c8 |= (uint32_t)(c >= 0x80u && c <= 0x8Fu) << e;
    c9 |= (uint32_t)(c >= 0x80u && c <= 0x9Fu) << e;
    ca |= (uint32_t)(c >= 0xA0u && c <= 0xBFu) << e;
  }
  const uint32_t covered = (ge2 << 1) | (ge3 << 2) | (l4 << 3);  // continuation positions some lead byte claims
  uint32_t b = badlead | (cont & ~covered);
  b |= (ge2 & ~(cont >> 1)) | (ge3 & ~(cont >> 2)) | (l4 & ~(cont >> 3));
  // second-byte ranges: E0 A0..BF (overlong), ED 80..9F (surrogates), F0 90..BF (overlong), F4 80..8F (> U+10FFFF)
  b |= (e0 & ~(ca >> 1)) | (ed & ~(c9 >> 1)) | (f0 & ~((ca | (c9 & ~c8)) >> 1)) | (f4 & ~(c8 >> 1));
  const uint32_t valid = nvalid == 16 ? 0xFFFFu : (1u << nvalid) - 1u;
  keep = (~nul >> 3) & valid;
  start = (~nul & (nul << 1)) >> 3 & valid;
  bad = (b >> 3) & valid;
}

struct KeptStarts {  // scan element: kept bytes (x) and sample starts (y) before a tile
  unsigned long long x, y;
};
struct AddKeptStarts {
  __host__ __device__ KeptStarts operator()(const KeptStarts& a, const KeptStarts& b) const { return {a.x + b.x, a.y + b.y}; }
};

// S1: kept bytes and sample starts per tile; the lowest position where decoding fails (atomicMin into *bad_pos).
__global__ void __launch_bounds__(CRLF_BLOCK) corpus_count(const uint8_t* __restrict__ text, uint64_t N,
                                                           KeptStarts* __restrict__ tile_cnt,
                                                           unsigned long long* __restrict__ bad_pos) {
  __shared__ uint32_t ws[CRLF_BLOCK / 32];
  const uint64_t base = (uint64_t)blockIdx.x * CRLF_TILE + (uint64_t)threadIdx.x * CRLF_PER_THREAD;
  uint4 v;
  uint32_t keep, start, bad, nvalid;
  corpus_mask16(text, N, base, v, keep, start, bad, nvalid);
  if (bad) atomicMin(bad_pos, (unsigned long long)(base + __ffs(bad) - 1));
  uint32_t c = __popc(keep) | (__popc(start) << 16);  // a tile has at most 4096 kept bytes and 2048 starts
#pragma unroll
  for (int o = 16; o; o >>= 1) c += __shfl_xor_sync(0xFFFFFFFFu, c, o);
  if ((threadIdx.x & 31) == 0) ws[threadIdx.x >> 5] = c;
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t t = 0;
#pragma unroll
    for (int i = 0; i < CRLF_BLOCK / 32; i++) t += ws[i];
    tile_cnt[blockIdx.x] = {t & 0xFFFFu, t >> 16};
  }
}

// S2 (one thread, after the scan): words[0] = samples, words[1] = kept bytes, words[2] = the sample *bad_pos lies in
// (~0 = every sample is valid UTF-8).
__global__ void corpus_words(const uint8_t* __restrict__ text, const KeptStarts* __restrict__ prefix, uint64_t n_tiles,
                             const unsigned long long* __restrict__ bad_pos, unsigned long long* __restrict__ words) {
  if (threadIdx.x || blockIdx.x) return;
  words[0] = prefix[n_tiles].y;
  words[1] = prefix[n_tiles].x;
  const unsigned long long q = *bad_pos;
  unsigned long long s = ~0ull;
  if (q != ~0ull) {
    const uint64_t t0 = q / CRLF_TILE * CRLF_TILE;
    s = prefix[q / CRLF_TILE].y;
    for (uint64_t p = t0; p <= q; p++) s += text[p] != 0 && (p == 0 || text[p - 1] == 0);
    s -= 1;  // a failing byte is never NUL, so a sample starts at or before it
  }
  words[2] = s;
}

// S3: compaction of the kept bytes (tile_compact_store) and the offset of every sample (off[S] = kept bytes).
__global__ void __launch_bounds__(CRLF_BLOCK) corpus_scatter(const uint8_t* __restrict__ text, uint64_t N,
                                                             const KeptStarts* __restrict__ prefix, uint64_t n_tiles,
                                                             uint8_t* __restrict__ out, uint64_t* __restrict__ off) {
  __shared__ uint32_t ws[CRLF_BLOCK / 32];
  __shared__ __align__(16) uint8_t stage[CRLF_TILE + 32];
  const uint64_t base = (uint64_t)blockIdx.x * CRLF_TILE + (uint64_t)threadIdx.x * CRLF_PER_THREAD;
  uint4 v;
  uint32_t keep, start, bad, nvalid;
  corpus_mask16(text, N, base, v, keep, start, bad, nvalid);
  uint32_t total;
  const uint32_t o = block_exclusive_scan(__popc(keep) | (__popc(start) << 16), ws, &total);
  const KeptStarts tp = prefix[blockIdx.x];
  uint64_t s = tp.y + (o >> 16);
  for (uint32_t sb = start; sb; sb &= sb - 1) {
    const int i = __ffs(sb) - 1;
    off[s++] = tp.x + (o & 0xFFFFu) + __popc(keep & ((1u << i) - 1u));
  }
  if (blockIdx.x == n_tiles - 1 && threadIdx.x == 0) off[prefix[n_tiles].y] = prefix[n_tiles].x;
  tile_compact_store(v, ~keep & 0xFFFFu, nvalid, o & 0xFFFFu, tp.x, total & 0xFFFFu, stage, out);
}

// Output of tgx_encode_corpus: the ids narrowed to T and, when sep >= 0, sep after every sample (sample i's ids move
// to id_off[i] + i).  Blocks take 256 consecutive ids; each finds its rows by binary search inside the rows of its block.
template <class T>
__global__ void __launch_bounds__(256) corpus_finalize(const uint32_t* __restrict__ ids, const uint64_t* __restrict__ id_off,
                                                       uint64_t S, long long sep, T* __restrict__ out) {
  __shared__ uint64_t rows[2];
  const uint64_t n = id_off[S];
  for (uint64_t b0 = (uint64_t)blockIdx.x * 256; b0 < n; b0 += (uint64_t)gridDim.x * 256) {
    const uint64_t t = b0 + threadIdx.x;
    if (sep < 0) {
      if (t < n) out[t] = (T)ids[t];
      continue;
    }
    auto row_of = [&](uint64_t x, uint64_t lo, uint64_t hi) {  // last r in [lo, hi] with id_off[r] <= x
      while (lo < hi) {
        const uint64_t mid = (lo + hi + 1) >> 1;
        if (id_off[mid] <= x) lo = mid; else hi = mid - 1;
      }
      return lo;
    };
    __syncthreads();
    if (threadIdx.x == 0) {
      rows[0] = row_of(b0, 0, S - 1);
      rows[1] = row_of(min(b0 + 255, n - 1), rows[0], S - 1);
    }
    __syncthreads();
    if (t < n) out[t + row_of(t, rows[0], rows[1])] = (T)ids[t];
  }
  if (sep >= 0)
    for (uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r < S; r += (uint64_t)gridDim.x * blockDim.x)
      out[id_off[r + 1] + r] = (T)sep;
}

// units = samples
__global__ void units_from_samples(const uint64_t* __restrict__ off, uint64_t S, uint64_t* __restrict__ ustart,
                                   uint32_t* __restrict__ ulen, uint32_t* __restrict__ idx,
                                   uint64_t* __restrict__ proc_len) {
  uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= S) return;
  uint64_t a = off[s], b = off[s + 1];
  ustart[s] = a;
  ulen[s] = (uint32_t)(b - a);
  idx[s] = (uint32_t)s;
  if (proc_len) proc_len[s] = b - a;
}

// units = snippets: sample.as_bytes().chunks(snippet_len)  (src/prune.rs:83)
__global__ void snippet_counts(const uint64_t* __restrict__ off, uint64_t S, uint64_t snip,
                               unsigned long long* __restrict__ cnt) {
  uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= S) return;
  uint64_t n = off[s + 1] - off[s];
  cnt[s] = (n + snip - 1) / snip;
}
__global__ void units_from_snippets(const uint64_t* __restrict__ off, uint64_t S, uint64_t snip,
                                    const unsigned long long* __restrict__ first_unit,
                                    uint64_t* __restrict__ ustart, uint32_t* __restrict__ ulen,
                                    uint32_t* __restrict__ idx, uint32_t* __restrict__ unit_sample) {
  uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= S) return;
  uint64_t a = off[s], n = off[s + 1] - a;
  unsigned long long u = first_unit[s];
  for (uint64_t o = 0; o < n; o += snip, u++) {
    ustart[u] = a + o;
    ulen[u] = (uint32_t)min((unsigned long long)snip, (unsigned long long)(n - o));
    idx[u] = (uint32_t)u;
    unit_sample[u] = (uint32_t)s;
  }
}

// counts[0] = #units with len >= long_threshold, counts[1] = #units with len >= 1,
// counts[2] = #units with len >= lane_threshold (E-step: snippets below it run one lane each)
__global__ void split_sorted(const uint32_t* __restrict__ sorted_len, uint32_t U, uint32_t long_threshold,
                             uint32_t lane_threshold, uint32_t* __restrict__ counts) {
  if (threadIdx.x || blockIdx.x) return;
  auto first_below = [&](uint32_t thr) {  // descending order: first index with len < thr
    uint32_t lo = 0, hi = U;
    while (lo < hi) {
      uint32_t mid = (lo + hi) >> 1;
      if (sorted_len[mid] >= thr) lo = mid + 1; else hi = mid;
    }
    return lo;
  };
  counts[0] = first_below(long_threshold);
  counts[1] = first_below(1);
  counts[2] = first_below(lane_threshold);
}

// lowest unit index with non-zero status (and its payload)
__global__ void first_bad_unit(const int32_t* __restrict__ status, uint32_t U, unsigned long long* __restrict__ out) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < U && status[i] != 0) atomicMin(out, (unsigned long long)i);
}

// Device memory is cleared by a kernel, not by cudaMemsetAsync: a memset may be scheduled on a copy
// engine, where it queues behind the bulk D2H copy of the previous chunk (tgx_encode_batch).
__global__ void fill_bytes_kernel(unsigned char* __restrict__ p, unsigned long long n, unsigned int byte) {
  const unsigned int w = byte * 0x01010101u;
  const unsigned long long head = min(n, (unsigned long long)((16 - (reinterpret_cast<unsigned long long>(p) & 15)) & 15));
  const unsigned long long nvec = (n - head) >> 4;
  const unsigned long long tid = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  const unsigned long long nthr = (unsigned long long)gridDim.x * blockDim.x;
  uint4* v = reinterpret_cast<uint4*>(p + head);
  for (unsigned long long i = tid; i < nvec; i += nthr) v[i] = make_uint4(w, w, w, w);
  const unsigned long long tail0 = head + (nvec << 4);
  for (unsigned long long i = tid; i < head; i += nthr) p[i] = (unsigned char)byte;
  for (unsigned long long i = tail0 + tid; i < n; i += nthr) p[i] = (unsigned char)byte;
}

__global__ void copy_u32(const uint32_t* __restrict__ src, uint32_t* __restrict__ dst, uint64_t n) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = src[i];
}

__global__ void add_u64(unsigned long long* __restrict__ dst, const unsigned long long* __restrict__ src, uint64_t n) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] += src[i];
}

// pair-frequency pass (src/merge.rs:61-64): key[t] = ids[t-1] * V + ids[t]; the first token of every sample gets
// the sentinel V * V (sorted behind every real pair) by pair_keys_mark_starts, which runs afterwards.
__global__ void pair_keys(const uint32_t* __restrict__ ids, unsigned long long T, unsigned long long V,
                          unsigned long long* __restrict__ keys) {
  const unsigned long long t = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= T) return;
  keys[t] = t ? (unsigned long long)ids[t - 1] * V + ids[t] : V * V;
}
__global__ void pair_keys_mark_starts(const uint64_t* __restrict__ id_off, uint64_t S, unsigned long long V,
                                      unsigned long long* __restrict__ keys) {
  const uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= S) return;
  if (id_off[s] < id_off[s + 1]) keys[id_off[s]] = V * V;
}
// n_pairs = runs that are not the sentinel run (the sentinel, if present, is the last run of the sorted keys)
__global__ void pair_count_runs(const unsigned long long* __restrict__ uniq, const unsigned long long* __restrict__ num_runs,
                                unsigned long long V, unsigned long long* __restrict__ n_pairs) {
  if (threadIdx.x || blockIdx.x) return;
  unsigned long long n = *num_runs;
  if (n && uniq[n - 1] == V * V) n--;
  *n_pairs = n;
}
__global__ void pair_unpack(const unsigned long long* __restrict__ packed, unsigned long long n, unsigned long long V,
                            unsigned long long* __restrict__ out) {
  const unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const unsigned long long k = packed[i];
  out[i] = ((k / V) << 32) | (k % V);
}

}  // namespace tgxk

// =========================================================================================
// host side
// =========================================================================================
namespace {

using namespace tgxk;

struct Timer {
  cudaEvent_t a, b;
};

cudaError_t dev_fill(void* p, int byte, size_t n, cudaStream_t st) {
  if (!n) return cudaSuccess;
  const uint32_t blocks = (uint32_t)std::min<uint64_t>(std::max<uint64_t>(1, (n + 4095) / 4096), 148 * 8);
  fill_bytes_kernel<<<blocks, 256, 0, st>>>(reinterpret_cast<unsigned char*>(p), (unsigned long long)n, (unsigned int)byte & 0xFFu);
  return cudaGetLastError();
}

template <int G, bool DROP = false>
cudaError_t launch_viterbi(tgx_model* m, ViterbiParams p) {
  if (!p.u.count) return cudaSuccess;
  size_t smem = warp_smem_bytes(p.u.rows, p.u.W, G) * WPB;
  cudaError_t e = cudaFuncSetAttribute(viterbi_kernel<G, DROP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  uint32_t per_block = WPB * (32 / G);
  uint32_t blocks = (p.u.count + per_block - 1) / per_block;
  viterbi_kernel<G, DROP><<<blocks, WPB * 32, smem, m->w().stream>>>(p);
  m->w().stats.launches += 1;
  return cudaGetLastError();
}

template <int R, int HOT, int MAXT, bool DROP = false>
cudaError_t launch_viterbi_pair(tgx_model* m, PairParams p, DropInfo di = DropInfo()) {
  auto kernel = [] {
    if constexpr (DROP) return viterbi_pair_drop_kernel<R, HOT, MAXT>;
    else return viterbi_pair_kernel<R, HOT, MAXT>;
  }();
  constexpr int WG = 2 * R + 1;
  const size_t budget = (size_t)m->smem_optin;
  uint32_t groups = (uint32_t)std::min<size_t>({(budget - (size_t)p.hot_slots * 16) / pair_group_bytes(R),
                                                (size_t)(MAXT / (32 * WG)), (size_t)15});
  if (m->groups > 0) groups = std::min<uint32_t>(groups, (uint32_t)m->groups);
  groups = std::max<uint32_t>(1, std::min<uint32_t>(groups, (p.u.count + 1) / 2));
  p.groups = groups;
  const size_t smem = pair_smem_bytes(R, groups, p.hot_slots);
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  // whatever the tables leave of the 256 KB L1/shared array caches trie slots beyond the staged prefix
  e = cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout,
                           (int)std::min<size_t>(100, (smem + 1024) * 100 / (228 * 1024) + 1));
  if (e != cudaSuccess) return e;
  const uint32_t grid =
      (uint32_t)std::min<uint64_t>(((uint64_t)p.u.count + 2 * groups - 1) / (2 * groups),
                                   (uint64_t)(m->pair_grid_cap ? m->pair_grid_cap : (uint32_t)m->num_sms));
  if (!m->pair_grid_cap) {  // (algo 3 clears the counter before it forks: nothing may sit in front of this kernel on
                            //  its stream, or the spare team CTAs take the SMs that were left free for it)
    e = dev_fill(p.counter, 0, 4, m->w().stream);
    if (e != cudaSuccess) return e;
  }
  if constexpr (DROP) kernel<<<grid, groups * WG * 32, smem, m->w().stream>>>(p, di);
  else kernel<<<grid, groups * WG * 32, smem, m->w().stream>>>(p);
  m->w().stats.launches += 1;
  return cudaGetLastError();
}

// Two shapes (measured on B200, tools/probe.py, 1 GB / the 16 longest samples alone):
//   latency   5 groups, two trie levels in shared memory, 72 registers: 35.8 ms / 13.5 ms
//   throughput  6 groups (R = 2) with one staged level, 64 registers:    33.5 ms / 16.0 ms
// A batch is bound by its longest sample unless it is large, so the throughput shape is used from
// `wide_bytes` input bytes on (the chunks of the host entry point stay below it).
template <int R>
cudaError_t launch_viterbi_pair_r(tgx_model* m, PairParams p, uint64_t n_bytes, DropInfo di = DropInfo()) {
  const size_t cap = (size_t)m->smem_optin / 4;
  if (di.dropout > 0.0) {  // one shape with the keyed draw in the producers: 5 groups, 72 registers
    if ((size_t)m->da.hot[1] * 16 <= cap) {
      p.hot_slots = m->da.hot[1];
      return launch_viterbi_pair<2, 1, 800, true>(m, p, di);
    }
    p.hot_slots = 0;
    return launch_viterbi_pair<2, 0, 800, true>(m, p, di);
  }
  const bool wide = m->pair_shape == 2 || (m->pair_shape == 0 && n_bytes >= m->wide_bytes);
  const int levels = std::min(m->hot_levels, wide ? 1 : 2);
  if (levels >= 2 && (size_t)m->da.hot[2] * 16 <= cap) {
    p.hot_slots = m->da.hot[2];
    return wide ? launch_viterbi_pair<R, 2, 960>(m, p) : launch_viterbi_pair<R, 2, 800>(m, p);
  }
  if (levels >= 1 && (size_t)m->da.hot[1] * 16 <= cap) {
    p.hot_slots = m->da.hot[1];
    return wide ? launch_viterbi_pair<R, 1, 960>(m, p) : launch_viterbi_pair<R, 1, 800>(m, p);
  }
  p.hot_slots = 0;
  return wide ? launch_viterbi_pair<R, 0, 960>(m, p) : launch_viterbi_pair<R, 0, 800>(m, p);
}

cudaError_t launch_viterbi_g(tgx_model* m, int G, const ViterbiParams& p) {
  if (p.dropout > 0.0) return G >= 32 ? launch_viterbi<32, true>(m, p) : launch_viterbi<8, true>(m, p);
  switch (G) {
    case 1: return launch_viterbi<1>(m, p);
    case 2: return launch_viterbi<2>(m, p);
    case 4: return launch_viterbi<4>(m, p);
    case 8: return launch_viterbi<8>(m, p);
    case 16: return launch_viterbi<16>(m, p);
    default: return launch_viterbi<32>(m, p);
  }
}

template <int G, bool DROP = false>
cudaError_t launch_fb(tgx_model* m, FbParams p, bool backward, cudaStream_t st) {
  if (!p.u.count) return cudaSuccess;
  size_t smem = warp_smem_bytes(p.u.rows, p.u.W, G) * WPB;
  cudaError_t e;
  uint32_t per_block = WPB * (32 / G);
  uint32_t blocks = (p.u.count + per_block - 1) / per_block;
  if (!backward) {
    e = cudaFuncSetAttribute(fb_forward_kernel<G, DROP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    fb_forward_kernel<G, DROP><<<blocks, WPB * 32, smem, st>>>(p);
  } else {
    e = cudaFuncSetAttribute(fb_backward_kernel<G, false, DROP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    fb_backward_kernel<G, false, DROP><<<blocks, WPB * 32, smem, st>>>(p);
  }
  m->w().stats.launches += 1;
  return cudaGetLastError();
}

cudaError_t launch_fb_g(tgx_model* m, int G, const FbParams& p, bool backward, cudaStream_t st) {
  if (p.dropout > 0.0) return G >= 32 ? launch_fb<32, true>(m, p, backward, st) : launch_fb<4, true>(m, p, backward, st);
  switch (G) {
    case 1: return launch_fb<1>(m, p, backward, st);
    case 2: return launch_fb<2>(m, p, backward, st);
    case 4: return launch_fb<4>(m, p, backward, st);
    case 8: return launch_fb<8>(m, p, backward, st);
    case 16: return launch_fb<16>(m, p, backward, st);
    default: return launch_fb<32>(m, p, backward, st);
  }
}

inline uint32_t nblk(uint64_t n, uint32_t t) { return (uint32_t)((n + t - 1) / t); }


int check_model(tgx_model* m) {
  if (!m) return fail(TGX_ERR_INVALID, "null model");
  if (m->device < 0)
    return fail(TGX_ERR_NO_DEVICE, "model was created host-only (device = -1); there is no CPU compute path");
  CU(cudaSetDevice(m->device));
  (void)cudaGetLastError();  // a stale non-sticky error of an earlier call must not fail this one
  return TGX_OK;
}

// The `_dev` entry points take buffers the caller has (maybe) just produced on ITS stream, while the library works on
// streams of its own.  Contract (include/tokengeex_b200.h): work queued on the legacy default stream — where torch and
// plain CUDA runtime calls put it unless told otherwise — before the call is ordered before the library's kernels;
// callers on other streams synchronise them first.  Results are complete when the call returns.
int order_after_caller(tgx_model* m) {
  CU(cudaEventRecord(m->ev_caller, cudaStreamLegacy));
  CU(cudaStreamWaitEvent(m->w().stream, m->ev_caller, 0));
  return TGX_OK;
}

// Token hash of the emit kernel (max_token_len <= 16 only); in a rebuild, a vocabulary it cannot serve leaves
// hash.mask == 0 and emit walks the trie.  On failure nothing the model already holds has been touched.
// `built`: a token hash of this vocabulary that the caller has built already (beside the trie, on a thread of its own),
// with the builder's message in `built_err`; null = build it here.
int upload_aux_tables(tgx_model* m, const tgx::DoubleArray& da, const uint8_t* token_bytes, const uint64_t* token_offsets,
                      uint64_t V, uint32_t max_token_len, tgx::TokenHash* built = nullptr,
                      const std::string* built_err = nullptr) {
  (void)da;
  if (m->device < 0) return TGX_OK;
  cudaStream_t st = m->w().stream;
  tgx::TokenHash h;
  bool hash_ok = V != 0 && max_token_len >= 1 && max_token_len <= 16;
  if (hash_ok && built) {
    hash_ok = built_err->empty();
    if (hash_ok) h = std::move(*built);
  } else if (hash_ok) {
    // (model creation: every vocabulary of 1..16-byte tokens gets its hash unless two distinct tokens share their key
    //  under every seed, i.e. the key function is broken — reported, not hidden behind the trie walk.  A rebuild builds
    //  the hash beside the trie and must leave the model unchanged on failure, so it keeps the trie walk instead.)
    const std::string herr = tgx::build_token_hash(token_bytes, token_offsets, V, &h);
    if (!herr.empty()) return fail(TGX_ERR_UNSUPPORTED, herr);
  }
  if (hash_ok) CU(m->d_hash.reserve(h.slots.size() * sizeof(tgx::Slot)));
  m->hash.mask = 0;
  m->hash.slots.clear();
  m->have_rows = false;  // the match tables belong to the previous vocabulary: rebuilt on first use
  if (hash_ok) {
    CU(cudaMemcpyAsync(m->d_hash.p, h.slots.data(), h.slots.size() * sizeof(tgx::Slot), cudaMemcpyHostToDevice, st));
    CU(cudaStreamSynchronize(st));
    m->hash = std::move(h);
  }
  return TGX_OK;
}

// Match tables (trie_build.h: slots8 / rows / row_ids) of the current vocabulary on the device; built and uploaded on
// first use.  have_rows stays false for vocabularies they cannot serve (tokens longer than 16 bytes).
int ensure_match_tables(tgx_model* m) {
  if (m->have_rows || m->device < 0) return TGX_OK;
  if (!tgx::build_match_tables(&m->da).empty()) return TGX_OK;
  const tgx::DoubleArray& da = m->da;
  cudaStream_t st = m->w().stream;
  CU(m->d_trie8.reserve(da.slots8.size() * 8));
  CU(m->d_rows.reserve(da.rows.size() * 8 + 256));
  CU(m->d_rowids.reserve(da.row_ids.size() * 4 + 256));
  CU(cudaMemcpyAsync(m->d_trie8.p, da.slots8.data(), da.slots8.size() * 8, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(m->d_rows.p, da.rows.data(), da.rows.size() * 8, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(m->d_rowids.p, da.row_ids.data(), da.row_ids.size() * 4, cudaMemcpyHostToDevice, st));
  CU(m->d_pair2.reserve(da.pair2.size() * 8));
  CU(cudaMemcpyAsync(m->d_pair2.p, da.pair2.data(), da.pair2.size() * 8, cudaMemcpyHostToDevice, st));
  CU(cudaStreamSynchronize(st));
  m->have_rows = true;
  m->rows16 = (uint32_t)(da.rows.size() / 2);
  return TGX_OK;
}

// crlf on device: (d_text,d_off) -> (m->w().text2, m->w().off2).  N = total bytes.
int run_crlf(tgx_model* m, const uint8_t* d_text, const uint64_t* d_off, uint64_t S, uint64_t N) {
  cudaStream_t st = m->w().stream;
  uint64_t n_tiles = (N + CRLF_TILE - 1) / CRLF_TILE;
  CU(m->w().text2.reserve(N + 16));
  CU(m->w().off2.reserve((S + 1) * 8));
  CU(m->w().bitmap.reserve((N / 32 + 4) * 4));
  CU(m->w().blk.reserve((n_tiles + 1) * 8 * 2));
  CU(dev_fill(m->w().bitmap.p, 0, (N / 32 + 4) * 4, st));
  if (S > 1) {
    crlf_mark_starts<<<nblk(S, 256), 256, 0, st>>>(d_off, S, m->w().bitmap.as<uint32_t>());
    m->w().stats.launches += 1;
  }
  unsigned long long* removed = m->w().blk.as<unsigned long long>();
  unsigned long long* prefix = removed + n_tiles + 1;
  CU(dev_fill(removed, 0, (n_tiles + 1) * 8, st));
  if (n_tiles) {
    crlf_count<<<(uint32_t)n_tiles, CRLF_BLOCK, 0, st>>>(d_text, N, m->w().bitmap.as<uint32_t>(), removed);
    m->w().stats.launches += 1;
  }
  size_t tmp = 0;
  CU(cub::DeviceScan::ExclusiveSum(nullptr, tmp, removed, prefix, (int)(n_tiles + 1), st));
  CU(m->w().cubtmp.reserve(tmp));
  CU(cub::DeviceScan::ExclusiveSum(m->w().cubtmp.p, tmp, removed, prefix, (int)(n_tiles + 1), st));
  m->w().stats.launches += 2;
  if (n_tiles) {
    crlf_scatter<<<(uint32_t)n_tiles, CRLF_BLOCK, 0, st>>>(d_text, N, d_off, S, m->w().bitmap.as<uint32_t>(), prefix,
                                                          n_tiles, m->w().text2.as<uint8_t>(), m->w().off2.as<uint64_t>());
    m->w().stats.launches += 1;
  } else {
    CU(dev_fill(m->w().off2.p, 0, (S + 1) * 8, st));  // no bytes at all: every sample is empty
  }
  CU(cudaGetLastError());
  return TGX_OK;
}

// sort unit indices by length, descending: keys in m->w().ulen, values in m->w().vals_in -> m->w().vals_out
int sort_units(tgx_model* m, uint32_t U) {
  CU(m->w().keys_out.reserve((size_t)U * 4 + 4));
  CU(m->w().vals_out.reserve((size_t)U * 4 + 4));
  size_t tmp = 0;
  CU(cub::DeviceRadixSort::SortPairsDescending(nullptr, tmp, m->w().ulen.as<uint32_t>(), m->w().keys_out.as<uint32_t>(),
                                               m->w().vals_in.as<uint32_t>(), m->w().vals_out.as<uint32_t>(), (int)U, 0, 32,
                                               m->w().stream));
  CU(m->w().cubtmp.reserve(tmp));
  CU(cub::DeviceRadixSort::SortPairsDescending(m->w().cubtmp.p, tmp, m->w().ulen.as<uint32_t>(), m->w().keys_out.as<uint32_t>(),
                                               m->w().vals_in.as<uint32_t>(), m->w().vals_out.as<uint32_t>(), (int)U, 0, 32,
                                               m->w().stream));
  m->w().stats.launches += 4;
  return TGX_OK;
}

int read_words(tgx_model* m, const void* d0, const void* d1, unsigned long long* o0, unsigned long long* o1);

// match_kernel over the whole blob: m->w().rec[p] = record of start position p (tgx_match_kernels.cuh)
int run_match(tgx_model* m, const uint8_t* d_text, uint64_t N, const uint8_t* d_skip = nullptr) {
  cudaStream_t st = m->w().stream;
  CU(m->w().rec.reserve((N + 64) * 4));
  MatchParams mp;
  mp.text = d_text;
  mp.blob_end = d_text + N;
  mp.N = N;
  mp.trie8 = m->d_trie8.as<uint2>();
  mp.root_base = m->da.root_base;
  mp.rec = m->w().rec.as<uint32_t>();
  mp.skip = d_skip;
  mp.pair2 = m->d_pair2.as<uint2>();
  mp.slice = 0;
  const size_t budget = (size_t)std::min<int64_t>(m->match_stage_bytes, (int64_t)m->smem_optin - 1024);
  mp.staged = (uint32_t)std::min<size_t>(m->da.slots8.size(), budget / 8);
  const size_t smem = (size_t)mp.staged * 8;
  auto launch = [&](auto kernel, int ilp) -> cudaError_t {
    const uint32_t threads = (uint32_t)std::min(m->match_threads, mk_max_threads(ilp));
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    const uint64_t per_cta = (uint64_t)threads * ilp;
    const uint64_t want = (uint64_t)m->num_sms * (uint64_t)std::max(1, m->match_ctas_per_sm);
    const uint64_t rounds = std::max<uint64_t>(1, (N + per_cta * want - 1) / (per_cta * want));
    mp.slice = rounds * per_cta;
    const uint32_t grid = (uint32_t)((N + mp.slice - 1) / mp.slice);
    kernel<<<grid, threads, smem, st>>>(mp);
    return cudaGetLastError();
  };
  if (m->match_compact) {  // walks compacted inside their warp: 1024 threads, four starts per lane, the queues behind the trie
    const uint32_t threads = MK2_THREADS;
    const size_t qbytes = (size_t)(threads / 32) * 2 * MK2_Q * 8;
    const size_t budget2 = (size_t)std::min<int64_t>(m->match_stage_bytes, (int64_t)m->smem_optin - 1024 - (int64_t)qbytes);
    mp.staged = (uint32_t)std::min<size_t>(m->da.slots8.size(), budget2 / 8);
    const size_t smem2 = (size_t)mp.staged * 8 + qbytes;
    CU(cudaFuncSetAttribute(match2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2));
    const uint64_t per_cta = (uint64_t)threads * 4;
    const uint64_t want = (uint64_t)m->num_sms * (uint64_t)std::max(1, m->match_ctas_per_sm);
    const uint64_t rounds = std::max<uint64_t>(1, (N + per_cta * want - 1) / (per_cta * want));
    mp.slice = rounds * per_cta;
    match2_kernel<<<(uint32_t)((N + mp.slice - 1) / mp.slice), threads, smem2, st>>>(mp);
    CU(cudaGetLastError());
    m->w().stats.launches += 1;
    return TGX_OK;
  }
  CU(launch(match_kernel<4>, 4));
  m->w().stats.launches += 1;
  return TGX_OK;
}

// Viterbi over all samples: forward dp (back lengths) + backtrack (token-end marks).  On return
// m->w().mark holds the length of the token ending at every marked byte, m->w().ntok token counts,
// m->w().status per-sample status.
int run_viterbi(tgx_model* m, const uint8_t* d_text, const uint64_t* d_off, uint64_t S, uint64_t N,
                uint64_t* d_proc_len, bool with_dropout = false) {
  cudaStream_t st = m->w().stream;
  if (S >= (1ull << 32)) return fail(TGX_ERR_INVALID, "too many samples in one call (< 2^32)");
  uint32_t U = (uint32_t)S;
  const uint64_t n_tiles = (N + EM_TILE - 1) / EM_TILE;
  CU(m->w().ustart.reserve((size_t)U * 8 + 8));
  CU(m->w().ulen.reserve((size_t)U * 4 + 4));
  CU(m->w().vals_in.reserve((size_t)U * 4 + 4));
  CU(m->w().bp.reserve(N + 64));
  CU(m->w().mark.reserve(n_tiles * EM_TILE + 64));
  CU(m->w().ntok.reserve(((size_t)U + 1) * 8));
  CU(m->w().status.reserve((size_t)U * 4 + 4));
  CU(m->w().small.reserve(256));
  units_from_samples<<<nblk(U, 256), 256, 0, st>>>(d_off, S, m->w().ustart.as<uint64_t>(), m->w().ulen.as<uint32_t>(),
                                                  m->w().vals_in.as<uint32_t>(), d_proc_len);
  m->w().stats.launches += 1;
  int rc = sort_units(m, U);
  if (rc) return rc;
  uint32_t* counts = m->w().small.as<uint32_t>();
  uint32_t thr = (uint32_t)std::min<int64_t>(m->long_threshold, 0x7FFFFFFF);
  const uint32_t thr2 = (uint32_t)std::min<int64_t>(m->team_long_threshold, 0x7FFFFFFF);
  split_sorted<<<1, 32, 0, st>>>(m->w().keys_out.as<uint32_t>(), U, thr, thr2, counts);
  m->w().stats.launches += 1;
  CU(dev_fill(m->w().ntok.p, 0, ((size_t)U + 1) * 8, st));
  CU(dev_fill(m->w().status.p, 0, (size_t)U * 4 + 4, st));
  CU(dev_fill(m->w().mark.p, 0, n_tiles * EM_TILE, st));
  // (no host synchronisation here: every kernel below reads its unit range from `counts`)

  UnitParams u;
  u.text = d_text;
  u.unit_start = m->w().ustart.as<uint64_t>();
  u.unit_len = m->w().ulen.as<uint32_t>();
  u.order = m->w().vals_out.as<uint32_t>();
  u.trie = m->d_trie;
  u.root_base = m->da.root_base;
  u.rows = std::max<uint32_t>(1, m->da.max_token_len);
  u.W = u.rows + 1;
  u.counts = counts;
  u.first = 0;
  u.count = U;  // upper bound for the grids

  const double dropout = with_dropout ? m->dropout : 0.0;  // the frequency passes encode with dropout 0.0
  // with the draw: pair-CTA or lane-group kernels
  // automatic: the teams for the encode entry points only (`with_dropout` marks them) — the frequency passes of the EM
  // loop run once per rebuilt model, where building the match tables costs more than the teams save (measured at
  // 4 GB / 250k tokens: 0.204 against 0.148 s)
  const int algo_req = m->algo == 4 ? (with_dropout && N >= m->wide_bytes && u.rows <= 16 ? 3 : 2) : m->algo;
  if (!(dropout > 0.0) && (algo_req == 0 || algo_req == 3) && u.rows <= 16) {
    rc = ensure_match_tables(m);
    if (rc) return rc;
  }
  const int algo = dropout > 0.0 ? (algo_req == 1 ? 1 : 2) : ((algo_req == 0 || algo_req == 3) && !m->have_rows ? 2 : algo_req);
  m->w().algo_used = algo;
  m->w().side_used = false;
  uint32_t n_long = 0;  // algo 3: samples of at least team_long_threshold bytes (the one host wait in the middle of a call)
  if (algo == 3 && u.rows <= 16 && N && U) {
    unsigned long long w01 = 0, w23 = 0;
    rc = read_words(m, counts, counts + 2, &w01, &w23);
    if (rc) return rc;
    n_long = std::min<uint32_t>((uint32_t)w23, (uint32_t)(w01 >> 32));  // min(counts[2], counts[1])
  }
  CU(cudaEventRecord(m->w().ev[8], st));
  if ((algo == 0 || algo == 3) && u.rows <= 16 && N) {
    const uint8_t* d_skip = nullptr;
    if (algo == 3 && n_long && m->match_compact && m->match_skip) {
      // nobody reads the records inside the samples the pair-CTA kernel takes: match2_kernel writes row 0 there
      const size_t nb = (size_t)((N + 127) >> 7);
      CU(m->w().skip.reserve(nb + 64));
      CU(dev_fill(m->w().skip.p, 0, nb, st));
      mark_skip_kernel<<<nblk((uint64_t)n_long * 32, 256), 256, 0, st>>>(u.unit_start, u.unit_len, u.order, n_long,
                                                                        m->w().skip.as<uint8_t>());
      m->w().stats.launches += 1;
      d_skip = m->w().skip.as<uint8_t>();
    }
    rc = run_match(m, d_text, N, d_skip);
    if (rc) return rc;
  }
  CU(cudaEventRecord(m->w().ev[9], st));
  CU(cudaEventRecord(m->w().ev[0], st));  // [0]..[1]: the consumer of the match stream / the forward kernel
  if (algo == 3 && u.rows <= 16) {
    if (N && U) {
      // The samples of at least team_long_threshold bytes run on the pair-CTA kernel (16 lanes per sample: the shortest
      // chain per position) BESIDE the teams, on P SMs of their own: forked when match_kernel — which fills every SM —
      // has finished.  Measured: a side kernel that runs beside match_kernel only adds its time to it, and persistent
      // team CTAs on every SM keep the pair CTAs waiting until they exit; so the team kernel gets num_sms - P CTAs,
      // the pair kernel P (highest stream priority), and P more team CTAs wait on a lowest-priority stream for the SMs
      // the pair CTAs free.  P needs the number of long samples on the host: n_long was read above.
      // A pair CTA runs 10 chains (5 groups of two samples) and a chain takes its samples longest first, so P is sized
      // for `side_load` / 10 samples per chain: the batch's longest sample bounds the side kernel anyway (12.6 ms for
      // 262144 bytes), and the shorter long ones fit behind each other inside that time on fewer SMs.
      const uint32_t per_cta = (uint32_t)std::max(1, m->side_load);
      const uint32_t P = n_long ? std::min<uint32_t>((n_long + per_cta - 1) / per_cta, (uint32_t)m->num_sms * 2u / 3u) : 0u;
      unsigned int* ctr = m->w().small.as<unsigned int>() + 8;
      CU(dev_fill(ctr, 0, 8, st));
      CU(cudaEventRecord(m->w().ev_side_fork, st));
      if (P) {
        CU(cudaStreamWaitEvent(m->w().stream_side, m->w().ev_side_fork, 0));
        PairParams pp;
        pp.u = u;
        pp.u.part = 3;
        pp.u.count = n_long;
        pp.blob_end = d_text + N;
        pp.bp = m->w().bp.as<uint8_t>();
        pp.counter = ctr;
        pp.dbg = 0;
        m->w().side_used = true;
        CU(cudaEventRecord(m->w().ev[10], m->w().stream_side));
        {
          cudaStream_t keep = m->w().stream;
          m->w().stream = m->w().stream_side;
          m->pair_grid_cap = P;
          const int keep_groups = m->groups;
          if (m->side_groups > 0) m->groups = m->groups > 0 ? std::min(m->groups, m->side_groups) : m->side_groups;
          cudaError_t e = launch_viterbi_pair_r<2>(m, pp, 0);
          m->groups = keep_groups;
          m->pair_grid_cap = 0;
          m->w().stream = keep;
          CU(e);
        }
        CU(cudaEventRecord(m->w().ev[11], m->w().stream_side));
        CU(cudaEventRecord(m->w().ev_side_join, m->w().stream_side));
        CU(cudaStreamWaitEvent(m->w().stream_low, m->w().ev_side_fork, 0));
      }
      TeamParams tm;
      tm.u = u;
      tm.u.part = 4;
      tm.u.count = U - std::min(U, n_long);
      tm.rec = m->w().rec.as<uint32_t>();
      tm.rows = m->d_rows.as<double>();
      tm.bp = m->w().bp.as<uint8_t>();
      tm.counter = m->w().small.as<unsigned int>() + 9;
      const size_t budget = (size_t)std::min<int64_t>(m->team_hot_bytes, (int64_t)m->smem_optin - 1024);
      tm.hot16 = (uint32_t)std::max<size_t>(std::min<size_t>(m->rows16, budget / 16), std::min<size_t>(m->rows16, 9));  // (row 0 is always staged)
      const size_t smem = (size_t)tm.hot16 * 16;
      const uint32_t n_short = tm.u.count;
      if (n_short) {  // one launch on the compute stream (num_sms - P CTAs) and, when the pair kernel holds P SMs, one of P CTAs behind it
        constexpr uint32_t warps = TM_WARPS, per_warp = 8;
        CU(cudaFuncSetAttribute(viterbi_team_kernel<warps>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        const uint32_t ctas = ((n_short + per_warp - 1) / per_warp + warps - 1) / warps;
        const uint32_t g1 = std::max<uint32_t>(1, std::min<uint32_t>(ctas, (uint32_t)m->num_sms - P));
        viterbi_team_kernel<warps><<<g1, warps * 32, smem, st>>>(tm);
        m->w().stats.launches += 1;
        if (P && ctas > g1) {
          viterbi_team_kernel<warps><<<std::min<uint32_t>(ctas - g1, P), warps * 32, smem, m->w().stream_low>>>(tm);
          m->w().stats.launches += 1;
        }
        CU(cudaGetLastError());
      }
      if (P) {
        CU(cudaEventRecord(m->w().ev_low_join, m->w().stream_low));
        CU(cudaStreamWaitEvent(st, m->w().ev_low_join, 0));
      }
    }
  } else if (algo == 0 && u.rows <= 16) {
    if (N && U) {
      RowsParams rp;
      rp.u = u;
      rp.u.part = 0;
      rp.rec = m->w().rec.as<uint32_t>();
      rp.rows = m->d_rows.as<double>();
      const size_t budget = (size_t)std::min<int64_t>(m->rows_hot_bytes, (int64_t)m->smem_optin - 1024);
      rp.hot16 = (uint32_t)std::min<size_t>(m->rows16, budget / 16);
      rp.bp = m->w().bp.as<uint8_t>();
      rp.counter = m->w().small.as<unsigned int>() + 8;
      const size_t smem = (size_t)rp.hot16 * 16;
      CU(cudaFuncSetAttribute(viterbi_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      CU(dev_fill(rp.counter, 0, 4, st));
      const uint32_t warps = (uint32_t)std::max(1, std::min(16, m->rows_warps));
      const uint32_t grid = (uint32_t)std::min<uint64_t>(((uint64_t)U + 2 * warps - 1) / (2 * warps), (uint64_t)m->num_sms);
      viterbi_rows_kernel<<<grid, warps * 32, smem, st>>>(rp);
      m->w().stats.launches += 1;
      CU(cudaGetLastError());
    }
  } else if (algo == 2 && u.rows <= 16) {
    PairParams p;
    p.u = u;
    p.u.part = 0;
    p.blob_end = d_text + N;
    p.bp = m->w().bp.as<uint8_t>();
    p.counter = m->w().small.as<unsigned int>() + 8;
    p.dbg = 0;
    DropInfo di;
    di.dropout = dropout;
    di.seed = m->drop_seed;
    di.unit_base = m->drop_unit_base;
    if (!p.u.count) {
    } else {
      CU(launch_viterbi_pair_r<2>(m, p, N, di));
    }
  } else {
    ViterbiParams p;
    p.u = u;
    p.bp = m->w().bp.as<uint8_t>();
    p.dropout = dropout;
    p.drop_seed = m->drop_seed;
    p.unit_base = m->drop_unit_base;
    p.u.part = 1;
    CU(launch_viterbi_g(m, 32, p));
    p.u.part = 2;
    CU(launch_viterbi_g(m, m->g_short, p));
  }
  CU(cudaEventRecord(m->w().ev[1], st));
  if (m->w().side_used) CU(cudaStreamWaitEvent(st, m->w().ev_side_join, 0));
  CU(cudaEventRecord(m->w().ev[12], st));
  CU(cudaEventRecord(m->w().ev[2], st));
  if (U) {
    BacktrackParams b;
    b.unit_start = u.unit_start;
    b.unit_len = u.unit_len;
    b.order = u.order;
    b.counts = counts;
    b.first = 0;
    b.count = U;
    b.bp = m->w().bp.as<uint8_t>();
    b.mark = m->w().mark.as<uint8_t>();
    b.n_tokens = m->w().ntok.as<unsigned long long>();
    b.status = m->w().status.as<int32_t>();
    // long samples (sorted first): one warp each; short ones: one thread each
    b.part = 1;
    backtrack_warp_kernel<<<nblk(U, BW_WARPS), BW_WARPS * 32, 0, st>>>(b);
    b.part = 2;
    backtrack_thread_kernel<<<nblk(U, BT_THREADS), BT_THREADS, 0, st>>>(b);
    m->w().stats.launches += 2;
    CU(cudaGetLastError());
  }
  CU(cudaEventRecord(m->w().ev[3], st));
  return TGX_OK;
}

// Token ids (and/or frequencies) from the marks: count per tile, scan, emit.
int run_emit(tgx_model* m, const uint8_t* d_text, uint64_t N, uint32_t* d_ids, uint64_t ids_cap,
             unsigned long long* d_freq) {
  cudaStream_t st = m->w().stream;
  const uint64_t n_tiles = (N + EM_TILE - 1) / EM_TILE;
  CU(cudaEventRecord(m->w().ev[4], st));
  if (n_tiles) {
    CU(m->w().tilecnt.reserve((n_tiles + 1) * 16));
    unsigned long long* cnt = m->w().tilecnt.as<unsigned long long>();
    unsigned long long* prefix = cnt + n_tiles + 1;
    const uint32_t grid = (uint32_t)std::min<uint64_t>(n_tiles, (uint64_t)m->num_sms * 8);
    mark_count_kernel<<<grid, EM_BLOCK, 0, st>>>(m->w().mark.as<uint4>(), n_tiles, cnt);
    size_t tmp = 0;
    CU(cub::DeviceScan::ExclusiveSum(nullptr, tmp, cnt, prefix, (int)n_tiles, st));
    CU(m->w().cubtmp.reserve(tmp));
    CU(cub::DeviceScan::ExclusiveSum(m->w().cubtmp.p, tmp, cnt, prefix, (int)n_tiles, st));
    EmitParams e;
    e.mark = m->w().mark.as<uint4>();
    e.text = d_text;
    e.text_bytes = N;
    e.n_tiles = n_tiles;
    e.tile_prefix = prefix;
    e.trie = m->d_trie;
    e.root_base = m->da.root_base;
    e.ids = d_ids;
    e.cap = ids_cap;
    e.freq = d_freq;
    e.V = (uint32_t)m->V;
    const bool use_hash = m->emit_hash && m->hash.mask != 0;
    e.hash = use_hash ? m->d_hash.as<uint4>() : nullptr;
    e.hash_mask = use_hash ? m->hash.mask : 0;
    e.hash_seed = m->hash.seed;
    emit_kernel<<<grid, EM_BLOCK, d_freq ? EM_HOT * 4 : 0, st>>>(e);
    m->w().stats.launches += 4;
    CU(cudaGetLastError());
  }
  CU(cudaEventRecord(m->w().ev[5], st));
  return TGX_OK;
}

// Reads up to two device words once everything queued on the compute stream has finished, through
// the control stream (see tgx_model::stream_ctl); returns with both streams idle.
int read_words(tgx_model* m, const void* d0, const void* d1, unsigned long long* o0, unsigned long long* o1) {
  CU(cudaEventRecord(m->w().ev_ctl, m->w().stream));
  CU(cudaStreamWaitEvent(m->w().stream_ctl, m->w().ev_ctl, 0));
  if (d0) CU(cudaMemcpyAsync(m->w().h_words, d0, 8, cudaMemcpyDeviceToHost, m->w().stream_ctl));
  if (d1) CU(cudaMemcpyAsync(m->w().h_words + 1, d1, 8, cudaMemcpyDeviceToHost, m->w().stream_ctl));
  CU(cudaStreamSynchronize(m->w().stream_ctl));
  if (d0 && o0) *o0 = m->w().h_words[0];
  if (d1 && o1) *o1 = m->w().h_words[1];
  return TGX_OK;
}

int first_bad(tgx_model* m, uint32_t U, int64_t* out_idx, const void* extra = nullptr, unsigned long long* extra_out = nullptr) {
  unsigned long long* d = m->w().small.as<unsigned long long>() + 2;
  CU(dev_fill(d, 0xFF, 8, m->w().stream));
  if (U) {
    first_bad_unit<<<nblk(U, 256), 256, 0, m->w().stream>>>(m->w().status.as<int32_t>(), U, d);
    m->w().stats.launches += 1;
  }
  unsigned long long h = ~0ull;
  int rc = read_words(m, d, extra, &h, extra_out);
  if (rc) return rc;
  *out_idx = (h == ~0ull) ? -1 : (int64_t)h;
  return TGX_OK;
}

void finish_stats(tgx_model* m, int which) {
  float ms = 0;
  if (cudaEventElapsedTime(&ms, m->w().ev[0], m->w().ev[1]) == cudaSuccess) {
    if (which == 1) m->w().stats.viterbi_ms = ms;
    if (which == 2) m->w().stats.fwd_ms = ms;
  }
  if (which == 2 && cudaEventElapsedTime(&ms, m->w().ev[2], m->w().ev[3]) == cudaSuccess) m->w().stats.bwd_ms = ms;
  if (which == 1 && cudaEventElapsedTime(&ms, m->w().ev[2], m->w().ev[3]) == cudaSuccess) m->w().stats.back_ms = ms;
  if (which == 1 && cudaEventElapsedTime(&ms, m->w().ev[4], m->w().ev[5]) == cudaSuccess) m->w().stats.emit_ms = ms;
  if (which == 1 && cudaEventElapsedTime(&ms, m->w().ev[8], m->w().ev[9]) == cudaSuccess) m->w().stats.match_ms = ms;
  if (which == 1 && cudaEventElapsedTime(&ms, m->w().ev[8], m->w().ev[12]) == cudaSuccess) m->w().stats.forward_ms = ms;
  if (which == 1) m->w().stats.algo = m->w().algo_used;
  if (which == 1 && m->w().side_used && cudaEventElapsedTime(&ms, m->w().ev[10], m->w().ev[11]) == cudaSuccess) m->w().stats.side_ms = ms;
  if (cudaEventElapsedTime(&ms, m->w().ev[6], m->w().ev[7]) == cudaSuccess) m->w().stats.total_ms = ms;
  m->last_stats = m->w().stats;
}

}  // namespace

// =========================================================================================
// C ABI
// =========================================================================================
extern "C" {

const char* tgx_last_error(void) { return g_err.c_str(); }

int tgx_model_create(const uint8_t* token_bytes, const uint64_t* token_offsets, const double* scores,
                     uint64_t vocab_size, int device, tgx_model** out) {
  if (!out || !token_offsets || (!token_bytes && vocab_size && token_offsets[vocab_size]) || (!scores && vocab_size))
    return fail(TGX_ERR_INVALID, "null argument");
  std::unique_ptr<tgx_model> m(new tgx_model());
  std::string err = tgx::build_double_array(token_bytes, token_offsets, scores, vocab_size, &m->da);
  if (!err.empty()) return fail(TGX_ERR_UNSUPPORTED, err);
  m->V = vocab_size;
  m->V_built = vocab_size;
  m->device = device;
  if (device >= 0) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || device >= n)
      return fail(TGX_ERR_NO_DEVICE, "CUDA device " + std::to_string(device) + " not available");
    CU(cudaSetDevice(device));
    CU(cudaDeviceGetAttribute(&m->num_sms, cudaDevAttrMultiProcessorCount, device));
    CU(cudaDeviceGetAttribute(&m->smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device));
    CU(cudaMemcpyToSymbol(tgxk::c_exp_hdr, TGX_EXP_HDR, sizeof(TGX_EXP_HDR)));
    CU(cudaMemcpyToSymbol(tgxk::c_log_hdr, TGX_LOG_HDR, sizeof(TGX_LOG_HDR)));
    CU(cudaMemcpyToSymbol(tgxk::c_exp_tab, TGX_EXP_TAB, sizeof(TGX_EXP_TAB)));
    CU(cudaMemcpyToSymbol(tgxk::c_log_tab, TGX_LOG_TAB, sizeof(TGX_LOG_TAB)));
    for (auto& w : m->ws) {
      CU(cudaStreamCreateWithFlags(&w.stream, cudaStreamNonBlocking));
      CU(cudaStreamCreateWithFlags(&w.stream_ctl, cudaStreamNonBlocking));
      CU(cudaEventCreateWithFlags(&w.ev_ctl, cudaEventDisableTiming));
      {  // forked when match_kernel has finished: pair CTAs first, then the teams, then the spare team CTAs
        int lo = 0, hi = 0;
        CU(cudaDeviceGetStreamPriorityRange(&lo, &hi));
        CU(cudaStreamCreateWithPriority(&w.stream_side, cudaStreamNonBlocking, hi));
        CU(cudaStreamCreateWithPriority(&w.stream_low, cudaStreamNonBlocking, lo));
      }
      CU(cudaEventCreateWithFlags(&w.ev_low_join, cudaEventDisableTiming));
      CU(cudaEventCreateWithFlags(&w.ev_side_fork, cudaEventDisableTiming));
      CU(cudaEventCreateWithFlags(&w.ev_side_join, cudaEventDisableTiming));
      CU(cudaHostAlloc(reinterpret_cast<void**>(&w.h_words), 64, cudaHostAllocDefault));
      for (auto& e : w.ev) CU(cudaEventCreate(&e));
    }
    CU(cudaStreamCreateWithFlags(&m->stream2, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&m->stream3, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&m->stream4, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&m->stream5, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&m->stream6, cudaStreamNonBlocking));
    CU(cudaEventCreateWithFlags(&m->ev_join6, cudaEventDisableTiming));
    for (auto& e : m->ev_grp) CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&m->ev_join5, cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&m->ev_join3, cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&m->ev_join4, cudaEventDisableTiming));
    CU(cudaStreamCreateWithFlags(&m->stream_h2d, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&m->stream_d2h, cudaStreamNonBlocking));
    for (int i = 0; i < 2; i++) {
      CU(cudaEventCreateWithFlags(&m->ev_h2d[i], cudaEventDisableTiming));
      CU(cudaEventCreateWithFlags(&m->ev_d2h[i], cudaEventDisableTiming));
      for (auto& e : m->ev_split[i]) CU(cudaEventCreate(&e));
    }
    CU(cudaEventCreateWithFlags(&m->ev_fork, cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&m->ev_join, cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&m->ev_caller, cudaEventDisableTiming));
    size_t bytes = m->da.slots.size() * sizeof(tgx::Slot);
    CU(cudaMalloc(&m->d_trie, bytes));
    m->trie_cap = m->da.slots.size();
    CU(cudaMemcpyAsync(m->d_trie, m->da.slots.data(), bytes, cudaMemcpyHostToDevice, m->w().stream));
    CU(cudaStreamSynchronize(m->w().stream));
    int rc = upload_aux_tables(m.get(), m->da, token_bytes, token_offsets, vocab_size, m->da.max_token_len);
    if (rc) return rc;
  }
  *out = m.release();
  return TGX_OK;
}

int tgx_model_rebuild(tgx_model* m, const uint8_t* token_bytes, const uint64_t* token_offsets, const double* scores,
                      uint64_t vocab_size) {
  if (!m || !token_offsets || (!token_bytes && vocab_size && token_offsets[vocab_size]) || (!scores && vocab_size))
    return fail(TGX_ERR_INVALID, "null argument");
  std::lock_guard<std::recursive_mutex> g(m->mu);
  // the token hash of the new vocabulary (what emit_kernel probes) only needs the bytes: built beside the trie
  tgx::TokenHash hash;
  std::string hash_err = "not built";
  std::thread hash_thread;
  if (m->device >= 0 && vocab_size)
    hash_thread = std::thread([&] { hash_err = tgx::build_token_hash(token_bytes, token_offsets, vocab_size, &hash); });
  struct Joiner {
    std::thread& t;
    ~Joiner() {
      if (t.joinable()) t.join();
    }
  } joiner{hash_thread};
  tgx::DoubleArray fresh;
  std::string err = "miss";
  // a subset of the vocabulary the array was built for, not much smaller than it: keep the layout (trie_build.h);
  // in place — a miss leaves the array untouched
  if (m->retarget_permille > 0 && m->V_built && vocab_size * 1000ull >= m->V_built * (uint64_t)m->retarget_permille)
    err = tgx::retarget_double_array(&m->da, token_bytes, token_offsets, scores, vocab_size);
  const bool in_place = err.empty();
  if (err == "miss") {
    err = tgx::build_double_array(token_bytes, token_offsets, scores, vocab_size, &fresh, /*hot_order=*/false);
    if (err.empty()) m->V_built = vocab_size;
  }
  if (!err.empty()) return fail(TGX_ERR_UNSUPPORTED, err);  // the model is unchanged
  if (!in_place) m->da = std::move(fresh);
  m->V = vocab_size;
  const tgx::DoubleArray& da = m->da;
  if (m->device >= 0) {
    CU(cudaSetDevice(m->device));
    CU(cudaStreamSynchronize(m->w().stream));
    if (da.slots.size() > m->trie_cap) {
      uint4* p = nullptr;
      CU(cudaMalloc(&p, da.slots.size() * sizeof(tgx::Slot)));
      if (m->d_trie) cudaFree(m->d_trie);
      m->d_trie = p;
      m->trie_cap = da.slots.size();
    }
    CU(cudaMemcpyAsync(m->d_trie, da.slots.data(), da.slots.size() * sizeof(tgx::Slot), cudaMemcpyHostToDevice, m->w().stream));
    CU(cudaStreamSynchronize(m->w().stream));
    if (hash_thread.joinable()) hash_thread.join();
    int rc = upload_aux_tables(m, da, token_bytes, token_offsets, vocab_size, da.max_token_len, &hash, &hash_err);
    if (rc) return rc;
  }
  return TGX_OK;
}

void tgx_model_destroy(tgx_model* m) {
  if (!m) return;
  if (m->device >= 0) {
    cudaSetDevice(m->device);
    cudaDeviceSynchronize();
    m->Bbeta.release();
    m->accfix.release();
    DevBuf* bufs[] = {&m->text, &m->off, &m->idoff, &m->A, &m->expected, &m->freq, &m->ids, &m->scount, &m->hot,
                      &m->text_b, &m->off_b, &m->ids_b, &m->idoff_b, &m->scount_b};
    for (auto* b : bufs) b->release();
    for (auto& w : m->ws) {
      DevBuf* wb[] = {&w.text2, &w.off2, &w.bitmap, &w.blk, &w.ustart, &w.ulen, &w.keys_out, &w.vals_in, &w.vals_out,
                      &w.cubtmp, &w.bp, &w.mark, &w.tilecnt, &w.ntok, &w.status, &w.small, &w.rec};
      for (auto* b : wb) b->release();
      for (auto& e : w.ev)
        if (e) cudaEventDestroy(e);
      if (w.stream) cudaStreamDestroy(w.stream);
      if (w.stream_ctl) cudaStreamDestroy(w.stream_ctl);
      if (w.ev_ctl) cudaEventDestroy(w.ev_ctl);
      if (w.stream_side) cudaStreamDestroy(w.stream_side);
      if (w.stream_low) cudaStreamDestroy(w.stream_low);
      if (w.ev_low_join) cudaEventDestroy(w.ev_low_join);
      if (w.ev_side_fork) cudaEventDestroy(w.ev_side_fork);
      if (w.ev_side_join) cudaEventDestroy(w.ev_side_join);
      if (w.h_words) cudaFreeHost(w.h_words);
    }
    if (m->d_trie) cudaFree(m->d_trie);
    m->d_hash.release();
    m->d_trie8.release();
    m->d_rows.release();
    m->d_pair2.release();
    m->d_rowids.release();
    if (m->stream2) cudaStreamDestroy(m->stream2);
    if (m->stream3) cudaStreamDestroy(m->stream3);
    if (m->stream4) cudaStreamDestroy(m->stream4);
    if (m->stream5) cudaStreamDestroy(m->stream5);
    if (m->stream6) cudaStreamDestroy(m->stream6);
    if (m->ev_join6) cudaEventDestroy(m->ev_join6);
    for (auto& e : m->ev_grp)
      if (e) cudaEventDestroy(e);
    if (m->ev_join5) cudaEventDestroy(m->ev_join5);
    if (m->ev_join3) cudaEventDestroy(m->ev_join3);
    if (m->ev_join4) cudaEventDestroy(m->ev_join4);
    if (m->stream_h2d) cudaStreamDestroy(m->stream_h2d);
    if (m->stream_d2h) cudaStreamDestroy(m->stream_d2h);
    for (int i = 0; i < 2; i++) {
      if (m->ev_h2d[i]) cudaEventDestroy(m->ev_h2d[i]);
      if (m->ev_d2h[i]) cudaEventDestroy(m->ev_d2h[i]);
      for (auto& e : m->ev_split[i])
        if (e) cudaEventDestroy(e);
      m->raw[i].release();
      m->split[i].release();
      m->fin[i].release();
    }
    if (m->h_off) cudaFreeHost(m->h_off);
    if (m->h_out) cudaFreeHost(m->h_out);
    if (m->ev_fork) cudaEventDestroy(m->ev_fork);
    if (m->ev_join) cudaEventDestroy(m->ev_join);
    if (m->ev_caller) cudaEventDestroy(m->ev_caller);
    (void)cudaGetLastError();  // nothing above is allowed to leak an error into the next call
  }
  delete m;
}

int tgx_model_get_info(const tgx_model* m, tgx_model_info* info) {
  if (!m || !info) return fail(TGX_ERR_INVALID, "null argument");
  info->vocab_size = m->V;
  info->max_token_len = m->da.max_token_len;
  info->trie_nodes = m->da.n_nodes;
  info->trie_slots = (uint32_t)m->da.slots.size();
  info->trie_terminals = m->da.n_terminals;
  info->device = m->device;
  return TGX_OK;
}

int tgx_model_common_prefix_search(const tgx_model* m, const uint8_t* text, uint64_t n, uint32_t* ids,
                                   uint32_t* lens, uint64_t cap, uint64_t* count) {
  if (!m || (!text && n) || !count) return fail(TGX_ERR_INVALID, "null argument");
  uint64_t k = 0;
  tgx::da_common_prefix_search(m->da, text, (size_t)n, [&](uint32_t id, uint32_t len) {
    if (k < cap) {
      if (ids) ids[k] = id;
      if (lens) lens[k] = len;
    }
    k++;
  });
  *count = k;
  return TGX_OK;
}

int tgx_model_set_option(tgx_model* m, int key, int64_t value) {
  if (!m) return fail(TGX_ERR_INVALID, "null model");
  auto okg = [](int64_t g) { return g == 1 || g == 2 || g == 4 || g == 8 || g == 16 || g == 32; };
  switch (key) {
    case 0: if (!okg(value)) return fail(TGX_ERR_INVALID, "lanes per sample must be 1,2,4,8,16,32"); m->g_short = (int)value; break;
    case 1: if (value < 1) return fail(TGX_ERR_INVALID, "threshold must be >= 1"); m->long_threshold = value; break;
    case 2: if (!okg(value)) return fail(TGX_ERR_INVALID, "lanes per snippet must be 1,2,4,8,16,32"); m->g_estep = (int)value; break;
    case 5: if (value < 0) return fail(TGX_ERR_INVALID, "threshold must be >= 0 (0 = automatic)"); m->estep_long_threshold = value; break;
    case 3: if (value < 0 || value > 4) return fail(TGX_ERR_INVALID, "algo must be 0..4"); m->algo = (int)value; break;
    case 32: if (value < 1) return fail(TGX_ERR_INVALID, "threshold must be >= 1"); m->team_long_threshold = value; break;
    case 45: if (value < 0 || value > 1000) return fail(TGX_ERR_INVALID, "per mille"); m->retarget_permille = (int)value; break;
    case 43: if (value < 0 || value > 15) return fail(TGX_ERR_INVALID, "groups per CTA must be 0..15"); m->side_groups = (int)value; break;
    case 39: m->match_skip = value ? 1 : 0; break;
    case 38: if (value < 1 || value > 1000) return fail(TGX_ERR_INVALID, "samples per CTA must be 1..1000"); m->side_load = (int)value; break;
    case 37: m->match_compact = value ? 1 : 0; break;
    case 35: if (value < 0) return fail(TGX_ERR_INVALID, "bytes must be >= 0"); m->team_hot_bytes = value; break;
    case 33: if (value < 1 || value > 64) return fail(TGX_ERR_INVALID, "CTAs per SM must be 1..64"); m->match_ctas_per_sm = (int)value; break;
    case 16: m->emit_hash = value ? 1 : 0; break;
    case 17: m->estep_lane_threshold = value; break;  // < 0 = automatic, 0 = off
    case 19: if (value < 0 || value > 2) return fail(TGX_ERR_INVALID, "E-step form must be 0..2"); m->estep_split = value ? 1 : 0; m->estep_rows = (int)value; break;
    case 20: if (value < 1 || value > 4096) return fail(TGX_ERR_INVALID, "replicas must be 1..4096"); m->hot_r = (int)value; break;
    case 21: if (value < 0 || value > (1 << 20)) return fail(TGX_ERR_INVALID, "hot ids must be 0..2^20"); m->hot_k = (int)value; break;
    case 18: if (value < 0 || value > 16) return fail(TGX_ERR_INVALID, "blocks per SM must be 0..16"); m->lane_blocks_per_sm = (int)value; break;
    case 11: m->overlap_chunks = value ? 1 : 0; break;
    case 14: if (value < 0 || value > 2) return fail(TGX_ERR_INVALID, "pair shape must be 0..2"); m->pair_shape = (int)value; break;
    case 13: if (value < 0 || value > 2) return fail(TGX_ERR_INVALID, "hot levels must be 0..2"); m->hot_levels = (int)value; break;
    case 7: if (value < 4096) return fail(TGX_ERR_INVALID, "chunk bytes must be >= 4096"); m->chunk_bytes = (uint64_t)value; break;
    case 22: if (value < 0) return fail(TGX_ERR_INVALID, "byte base must be >= 0"); m->drop_byte_base = (uint64_t)value; break;
    case 23: if (value < 32 || value > 1024 || value % 32) return fail(TGX_ERR_INVALID, "match threads must be 32..1024, a multiple of 32"); m->match_threads = (int)value; break;
    case 24: if (value < 0) return fail(TGX_ERR_INVALID, "bytes must be >= 0"); m->match_stage_bytes = value; break;
    case 25: if (value < 1 || value > 32) return fail(TGX_ERR_INVALID, "warps must be 1..32"); m->rows_warps = (int)value; break;
    case 26: if (value < 0) return fail(TGX_ERR_INVALID, "bytes must be >= 0"); m->rows_hot_bytes = value; break;
    case 30: if (value < 0 || value > 1000) return fail(TGX_ERR_INVALID, "per mille"); m->estep_cut1 = (int)value; break;
    case 31: if (value < 0 || value > 1000) return fail(TGX_ERR_INVALID, "per mille"); m->estep_cut2 = (int)value; break;
    case 6: if (value < 0 || value > 15) return fail(TGX_ERR_INVALID, "groups per CTA must be 0..15"); m->groups = (int)value; break;
    default: return fail(TGX_ERR_INVALID, "unknown option");
  }
  return TGX_OK;
}

int tgx_model_set_dropout(tgx_model* m, double dropout, uint64_t seed) {
  if (!m) return fail(TGX_ERR_INVALID, "null model");
  if (!(dropout >= 0.0) || dropout >= 1.0)
    return fail(TGX_ERR_INVALID, "dropout must be in [0, 1): dropout >= 1 is a bytes-only vocabulary, not a draw");
  std::lock_guard<std::recursive_mutex> g(m->mu);
  m->dropout = dropout;
  m->drop_seed = seed;
  return TGX_OK;
}

double tgx_model_last_stat(const tgx_model* m, int what) {
  if (!m) return 0;
  switch (what) {
    case 0: return m->last_stats.launches;
    case 1: return m->last_stats.viterbi_ms;
    case 2: return m->last_stats.fwd_ms;
    case 3: return m->last_stats.bwd_ms;
    case 4: return m->last_stats.total_ms;
    case 5: return m->last_stats.back_ms;
    case 6: return m->last_stats.emit_ms;
    case 7: return m->last_stats.match_ms;
    case 8: return m->last_stats.forward_ms;  // match + consumers (+ the wait for the side stream)
    case 10: return m->last_stats.algo;       // forward algorithm the call used (option 3; 4 = automatic resolves to 2 or 3)
    case 9: return m->last_stats.side_ms;     // pair-CTA kernel of the longest samples on the side stream (algo 3)
    case 11: return m->last_stats.split_ms;   // tgx_encode_corpus: split kernels of every chunk
  }
  return 0;
}

int tgx_model_prune_select(tgx_model* m, const uint8_t* token_bytes, const uint64_t* token_offsets, const double* scores,
                           const uint8_t* keep, uint64_t vocab_size, const uint64_t* freq, uint64_t n_samples,
                           uint64_t target_vocab_size, double shrink_factor, int threads, uint32_t* out_ids,
                           uint64_t* out_n, double* audit) {
  if (!m) return fail(TGX_ERR_INVALID, "null model");
  std::lock_guard<std::recursive_mutex> g(m->mu);
  if (vocab_size != m->V) return fail(TGX_ERR_INVALID, "vocabulary is not the one the model was built from");
  int rc = tgx::prune_select_with(m->da, token_bytes, token_offsets, scores, keep, vocab_size, freq, n_samples,
                                  target_vocab_size, shrink_factor, threads, out_ids, out_n, audit);
  if (rc) return fail(rc, "prune_vocab failed (loss is not normal, or bad argument)");
  return TGX_OK;
}

// Developer aid (tools/analyse_rows.py; not part of include/tokengeex_b200.h): host walk of the 8-byte trie from every
// byte of `text`.  out[0] = probes, out[1] = probes of slots below `staged` (what match_kernel would serve from shared
// memory), out[2] = positions, out[3] = matches.
int tgx_debug_probe_stats(tgx_model* m, const uint8_t* text, uint64_t n, uint32_t staged, uint64_t* out) {
  if (!m || !text || !out || !tgx::build_match_tables(&m->da).empty()) return fail(TGX_ERR_INVALID, "no match tables");
  uint64_t probes = 0, low = 0, matches = 0;
  for (uint64_t p = 0; p < n; p++) {
    uint32_t xb = m->da.root_base;
    for (uint64_t d = 0; d < 16 && p + d < n; d++) {
      const uint32_t cw = 0x100u | text[p + d];
      const uint32_t t = xb ^ cw;
      probes++;
      if (t < staged) low++;
      if (t >= m->da.slots8.size()) break;
      const uint64_t e = m->da.slots8[t];
      const uint32_t ex = (uint32_t)e, ey = (uint32_t)(e >> 32);
      if ((ex ^ cw) & 0x1FFu) break;
      if (ey & tgx::SLOT8_TERM) matches++;
      if (!(ey & tgx::SLOT8_HASCH)) break;
      xb = ex >> 9;
    }
  }
  out[0] = probes; out[1] = low; out[2] = n; out[3] = matches;
  return TGX_OK;
}

int tgx_host_alloc(void** p, uint64_t bytes) {
  if (!p) return fail(TGX_ERR_INVALID, "null argument");
  CU(cudaHostAlloc(p, bytes ? bytes : 1, cudaHostAllocDefault));
  return TGX_OK;
}
int tgx_host_free(void* p) {
  if (p) CU(cudaFreeHost(p));
  return TGX_OK;
}

// ---------------------------------------------------------------------------- crlf
int tgx_crlf_batch(tgx_model* m, const uint8_t* text, const uint64_t* off, uint64_t S, uint8_t* out_text,
                   uint64_t* out_off) {
  int rc = check_model(m);
  if (rc) return rc;
  if (!off || !out_off || off[0] != 0) return fail(TGX_ERR_INVALID, "offsets must start at 0");
  std::lock_guard<std::recursive_mutex> g(m->mu);
  m->w().stats = Stats();
  uint64_t N = off[S];
  CU(m->text.reserve(N + 16));
  CU(m->off.reserve((S + 1) * 8));
  CU(cudaMemcpyAsync(m->text.p, text, N, cudaMemcpyHostToDevice, m->w().stream));
  CU(cudaMemcpyAsync(m->off.p, off, (S + 1) * 8, cudaMemcpyHostToDevice, m->w().stream));
  rc = run_crlf(m, m->text.as<uint8_t>(), m->off.as<uint64_t>(), S, N);
  if (rc) return rc;
  CU(cudaMemcpyAsync(out_off, m->w().off2.p, (S + 1) * 8, cudaMemcpyDeviceToHost, m->w().stream));
  CU(cudaStreamSynchronize(m->w().stream));
  CU(cudaMemcpyAsync(out_text, m->w().text2.p, out_off[S], cudaMemcpyDeviceToHost, m->w().stream));
  CU(cudaStreamSynchronize(m->w().stream));
  return TGX_OK;
}

// ---------------------------------------------------------------------------- encode
namespace {

// Queues every kernel of one encode batch on the current workspace; nothing here waits for the device.
int encode_enqueue(tgx_model* m, const uint8_t* d_text, const uint64_t* d_off, uint64_t S, uint64_t n_bytes,
                   uint32_t flags, uint32_t* d_ids, uint64_t ids_cap, uint64_t* d_id_off, int32_t* d_status,
                   uint64_t* d_proc_len, bool with_dropout = false) {
  m->w().stats = Stats();
  cudaStream_t st = m->w().stream;
  CU(cudaEventRecord(m->w().ev[6], st));
  const uint8_t* text = d_text;
  const uint64_t* off = d_off;
  int rc;
  if (flags & TGX_FLAG_CRLF) {
    rc = run_crlf(m, d_text, d_off, S, n_bytes);
    if (rc) return rc;
    text = m->w().text2.as<uint8_t>();
    off = m->w().off2.as<uint64_t>();
  }
  rc = run_viterbi(m, text, off, S, n_bytes, d_proc_len, with_dropout);
  if (rc) return rc;
  // id offsets = exclusive scan of token counts (S+1 entries; ntok[S] was zeroed)
  size_t tmp = 0;
  CU(cub::DeviceScan::ExclusiveSum(nullptr, tmp, m->w().ntok.as<unsigned long long>(),
                                   reinterpret_cast<unsigned long long*>(d_id_off), (int)(S + 1), st));
  CU(m->w().cubtmp.reserve(tmp));
  CU(cub::DeviceScan::ExclusiveSum(m->w().cubtmp.p, tmp, m->w().ntok.as<unsigned long long>(),
                                   reinterpret_cast<unsigned long long*>(d_id_off), (int)(S + 1), st));
  m->w().stats.launches += 2;
  rc = run_emit(m, text, n_bytes, d_ids, ids_cap, nullptr);
  if (rc) return rc;
  if (d_status) {  // (a kernel, not a D2D memcpy: keep the compute stream off the copy engines)
    copy_u32<<<nblk(S, 256), 256, 0, st>>>(reinterpret_cast<const uint32_t*>(m->w().status.p),
                                           reinterpret_cast<uint32_t*>(d_status), S);
    m->w().stats.launches += 1;
  }
  // control words: lowest failing sample and the total id count, read through the control stream
  unsigned long long* d = m->w().small.as<unsigned long long>() + 2;
  CU(dev_fill(d, 0xFF, 8, st));
  first_bad_unit<<<nblk(S, 256), 256, 0, st>>>(m->w().status.as<int32_t>(), (uint32_t)S, d);
  m->w().stats.launches += 1;
  CU(cudaEventRecord(m->w().ev[7], st));
  CU(cudaEventRecord(m->w().ev_ctl, st));
  CU(cudaStreamWaitEvent(m->w().stream_ctl, m->w().ev_ctl, 0));
  CU(cudaMemcpyAsync(m->w().h_words, d, 8, cudaMemcpyDeviceToHost, m->w().stream_ctl));
  CU(cudaMemcpyAsync(m->w().h_words + 1, d_id_off + S, 8, cudaMemcpyDeviceToHost, m->w().stream_ctl));
  return TGX_OK;
}

// Waits for the batch queued on the current workspace; total id count and lowest failing sample (-1 = none).
int encode_finish(tgx_model* m, uint64_t* total_ids, int64_t* bad) {
  CU(cudaStreamSynchronize(m->w().stream_ctl));
  CU(cudaStreamSynchronize(m->w().stream));
  finish_stats(m, 1);
  const unsigned long long h = m->w().h_words[0];
  *bad = (h == ~0ull) ? -1 : (int64_t)h;
  *total_ids = m->w().h_words[1];
  return TGX_OK;
}

}  // namespace

int tgx_encode_batch_dev(tgx_model* m, const uint8_t* d_text, const uint64_t* d_off, uint64_t S,
                         uint64_t n_bytes, uint32_t flags, uint32_t* d_ids, uint64_t ids_cap,
                         uint64_t* d_id_off, int32_t* d_status, uint64_t* d_proc_len, uint64_t* total_ids,
                         int64_t* first_bad_out) {
  int rc = check_model(m);
  if (rc) return rc;
  if (!d_off || !d_id_off || (!d_ids && ids_cap)) return fail(TGX_ERR_INVALID, "null argument");
  std::lock_guard<std::recursive_mutex> g(m->mu);
  if (first_bad_out) *first_bad_out = -1;
  if (total_ids) *total_ids = 0;
  if (S >= (1ull << 32)) return fail(TGX_ERR_INVALID, "too many samples in one call (< 2^32)");
  if (S == 0) {
    CU(dev_fill(d_id_off, 0, 8, m->w().stream));
    CU(cudaStreamSynchronize(m->w().stream));
    return TGX_OK;
  }
  m->drop_unit_base = 0;
  rc = encode_enqueue(m, d_text, d_off, S, n_bytes, flags, d_ids, ids_cap, d_id_off, d_status, d_proc_len, true);
  if (rc) return rc;
  uint64_t tot = 0;
  int64_t bad = -1;
  rc = encode_finish(m, &tot, &bad);
  if (rc) return rc;
  if (total_ids) *total_ids = tot;
  if (first_bad_out) *first_bad_out = bad;
  if (tot > ids_cap) return fail(TGX_ERR_CAPACITY, "ids capacity too small: need " + std::to_string(tot));
  if (bad >= 0) return fail(TGX_ERR_NO_PATH, "no path for sample " + std::to_string(bad));
  return TGX_OK;
}

namespace {

// ---- chunk pipeline of the host entry points (tgx_encode_batch, tgx_encode_corpus)
// Chunks of whole samples (~chunk_bytes each): the H2D copy of chunk k+1 and the D2H copy of chunk k-1 run on their own
// streams beside the kernels of chunk k (two buffer sets).  What reaches the device and what leaves it is the caller's:

// Input stage: puts chunk k's samples as blob + offsets into buffer set b (m->text / m->text_b, m->off / m->off_b).
struct ChunkInput {
  uint64_t K = 1;      // chunks
  uint64_t max_b = 0;  // bytes of the largest chunk as it reaches the device
  uint64_t max_s = 0;  // samples of the largest chunk, when known before the chunks are split
  virtual ~ChunkInput() = default;
  // Queues the H2D copy of chunk k on `st` (the copy-in stream when K > 1); returns without waiting.
  virtual int h2d(tgx_model* m, uint64_t k, int b, cudaStream_t st) = 0;
  // Queued on the compute stream of chunk k's workspace right after the copy was queued (so behind the previous
  // chunk's kernels); returns without waiting.
  virtual int after_h2d(tgx_model*, uint64_t, int) { return TGX_OK; }
  // Chunk k's first sample, sample count and text bytes once its blob + offsets are (queued to be) in set b.  May wait.
  virtual int samples(tgx_model* m, uint64_t k, int b, uint64_t* s0, uint64_t* S, uint64_t* n) = 0;
};

// Output stage: takes chunk k's ids (m->ids / m->ids_b), id offsets (chunk-relative) and per-sample status / length.
struct ChunkOutput {
  virtual ~ChunkOutput() = default;
  // Queued on the compute stream behind the chunk's encode kernels.
  virtual int after_encode(tgx_model*, uint64_t, int, uint64_t) { return TGX_OK; }
  // Queues the D2H copies of chunk k on `st` (its kernels have finished); `tot` ids, `base` ids in earlier chunks.
  // `bad` = the chunk's lowest sample without a path (-1 = none).
  virtual int d2h(tgx_model* m, uint64_t k, int b, uint64_t s0, uint64_t S, uint64_t tot, uint64_t base, int64_t bad,
                  const int32_t* d_status, const uint64_t* d_plen, cudaStream_t st) = 0;
};

DevBuf* set_text(tgx_model* m, int b) { return b ? &m->text_b : &m->text; }
DevBuf* set_off(tgx_model* m, int b) { return b ? &m->off_b : &m->off; }
DevBuf* set_ids(tgx_model* m, int b) { return b ? &m->ids_b : &m->ids; }
DevBuf* set_idoff(tgx_model* m, int b) { return b ? &m->idoff_b : &m->idoff; }
DevBuf* set_sc(tgx_model* m, int b) { return b ? &m->scount_b : &m->scount; }

// Runs the pipeline; *bad_all = lowest failing sample (-1 = none), *total = ids of all chunks, *stop = the input stage
// refused a chunk (its status; the chunks before it are encoded).  Returns with every copy finished.
int encode_chunks(tgx_model* m, uint32_t flags, uint64_t unit_base, ChunkInput& in, ChunkOutput& out,
                  int64_t* bad_all_out, uint64_t* total) {
  const uint64_t K = in.K;
  const int nset = K > 1 ? 2 : 1;
  for (int i = 0; i < nset; i++) {
    CU(set_text(m, i)->reserve(in.max_b + 16));
    CU(set_off(m, i)->reserve((in.max_s + 1) * 8));
    CU(set_ids(m, i)->reserve((in.max_b + 4) * 4));
    CU(set_idoff(m, i)->reserve((in.max_s + 1) * 8));
    CU(set_sc(m, i)->reserve((in.max_s + 1) * 12 + 32));
  }
  auto reserve_samples = [&](uint64_t k, int b, uint64_t Sk) -> int {  // (chunks split on the device only)
    if ((Sk + 1) * 8 <= set_idoff(m, b)->cap && (Sk + 1) * 12 + 32 <= set_sc(m, b)->cap) return TGX_OK;
    if (K > 1 && k >= 2) CU(cudaEventSynchronize(m->ev_d2h[b]));  // the set's previous results left the device
    CU(set_idoff(m, b)->reserve((Sk + 1) * 8));
    CU(set_sc(m, b)->reserve((Sk + 1) * 12 + 32));
    return TGX_OK;
  };
  std::vector<cudaEvent_t> tev;  // trace: [base, per chunk: h2d0,h2d1,c0,c1,d2h0,d2h1]
  const bool overlap = K > 1 && m->overlap_chunks;
  auto h2d = [&](uint64_t k) -> int {
    const int b = (int)(k & 1);
    cudaStream_t st = K > 1 ? m->stream_h2d : m->w().stream;
    if (!tev.empty()) cudaEventRecord(tev[1 + 6 * k + 0], st);
    int r = in.h2d(m, k, b, st);
    if (r) return r;
    if (!tev.empty()) cudaEventRecord(tev[1 + 6 * k + 1], st);
    if (K > 1) CU(cudaEventRecord(m->ev_h2d[b], st));
    const int wi = m->wi;
    m->wi = overlap ? b : 0;
    r = in.after_h2d(m, k, b);
    m->wi = wi;
    return r;
  };
  const bool trace = getenv("TGX_TRACE") != nullptr;
  auto now_ms = [] {
    timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6;
  };
  const double t_begin = now_ms();
  if (trace) {
    tev.resize(1 + 6 * K);
    for (auto& e : tev) cudaEventCreate(&e);
    cudaEventRecord(tev[0], m->w().stream);
  }
  // Pipeline over chunks k = 0..K-1 with two buffer sets and two workspaces (set / workspace k & 1):
  //   H2D(k+1) on the copy-in stream, kernels(k+1) QUEUED on the other workspace before the host waits for
  //   chunk k, D2H(k) on the copy-out stream.  Queuing the next chunk early lets its kernels take over the SMs
  //   that chunk k's forward kernel frees while its last long samples finish on a few SMs.
  std::vector<uint64_t> s0s(K, 0), Sks(K, 0), nbs(K, 0);
  auto enqueue = [&](uint64_t k) -> int {
    const int b = (int)(k & 1);
    m->wi = overlap ? b : 0;
    if (K > 1) {
      CU(cudaStreamWaitEvent(m->w().stream, m->ev_h2d[b], 0));
      if (k >= 2) CU(cudaStreamWaitEvent(m->w().stream, m->ev_d2h[b], 0));  // the set's previous results left the device
    }
    uint64_t s0 = 0, Sk = 0, nb = 0;
    int r = in.samples(m, k, b, &s0, &Sk, &nb);
    if (r) return r;
    s0s[k] = s0;
    Sks[k] = Sk;
    nbs[k] = nb;
    if (Sk >= (1ull << 32)) return fail(TGX_ERR_UNSUPPORTED, "too many samples in one chunk (< 2^32)");
    r = reserve_samples(k, b, Sk);
    if (r) return r;
    int32_t* dst = set_sc(m, b)->as<int32_t>();
    uint64_t* dpl = reinterpret_cast<uint64_t*>(set_sc(m, b)->as<unsigned char>() + ((Sk * 4 + 15) & ~15ull));
    if (!tev.empty()) cudaEventRecord(tev[1 + 6 * k + 2], m->w().stream);
    if (Sk == 0) return TGX_OK;
    m->drop_unit_base = unit_base + s0;  // the draw is keyed by the sample's index in the whole input, not in its chunk
    r = encode_enqueue(m, set_text(m, b)->as<uint8_t>(), set_off(m, b)->as<uint64_t>(), Sk, nb, flags,
                       set_ids(m, b)->as<uint32_t>(), nb + 4, set_idoff(m, b)->as<uint64_t>(), dst, dpl, true);
    if (r) return r;
    r = out.after_encode(m, k, b, Sk);
    if (r) return r;
    if (!tev.empty()) cudaEventRecord(tev[1 + 6 * k + 3], m->w().stream);
    return TGX_OK;
  };
  // (a failure below leaves copies in flight: callers' buffers are written until the streams drain)
  auto drain = [&](int rc) {
    if (K > 1) {
      cudaStreamSynchronize(m->stream_h2d);
      cudaStreamSynchronize(m->stream_d2h);
    }
    for (auto& w : m->ws) cudaStreamSynchronize(w.stream);
    for (auto& e : tev) cudaEventDestroy(e);
    return rc;
  };
  int rc = h2d(0);
  if (rc) return drain(rc);
  rc = enqueue(0);
  if (rc) return drain(rc);
  uint64_t base = 0;  // ids emitted by earlier chunks
  int64_t bad_all = -1;
  for (uint64_t k = 0; k < K; k++) {
    const int b = (int)(k & 1);
    if (k + 1 < K) {
      rc = h2d(k + 1);
      if (rc) return drain(rc);
      if (overlap) {
        rc = enqueue(k + 1);
        if (rc) return drain(rc);
      }
    }
    const uint64_t s0 = s0s[k], Sk = Sks[k];
    int32_t* dst = set_sc(m, b)->as<int32_t>();
    uint64_t* dpl = reinterpret_cast<uint64_t*>(set_sc(m, b)->as<unsigned char>() + ((Sk * 4 + 15) & ~15ull));
    uint64_t tot = 0;
    int64_t bad = -1;
    m->wi = overlap ? b : 0;
    if (Sk) {
      rc = encode_finish(m, &tot, &bad);
      if (rc) return drain(rc);
    }
    if (trace)
      fprintf(stderr, "[tgx] chunk %llu/%llu: kernels done at %.2f ms (device %.2f ms)\n", (unsigned long long)k,
              (unsigned long long)K, now_ms() - t_begin, m->last_stats.total_ms);
    if (tot > nbs[k] + 4) return drain(fail(TGX_ERR_CUDA, "internal: more ids than bytes"));
    if (bad >= 0 && bad_all < 0) bad_all = (int64_t)(s0 + bad);
    cudaStream_t st = K > 1 ? m->stream_d2h : m->w().stream;  // the chunk's kernels have finished
    if (!tev.empty()) cudaEventRecord(tev[1 + 6 * k + 4], st);
    rc = out.d2h(m, k, b, s0, Sk, tot, base, bad, dst, dpl, st);
    if (rc) return drain(rc);
    if (K > 1) CU(cudaEventRecord(m->ev_d2h[b], st));
    if (!tev.empty()) cudaEventRecord(tev[1 + 6 * k + 5], st);
    base += tot;
    if (!overlap && k + 1 < K) {
      rc = enqueue(k + 1);
      if (rc) return drain(rc);
    }
  }
  CU(cudaStreamSynchronize(K > 1 ? m->stream_d2h : m->w().stream));
  m->wi = 0;
  if (trace) {
    fprintf(stderr, "[tgx] all copies done at %.2f ms\n", now_ms() - t_begin);
    cudaDeviceSynchronize();
    for (uint64_t k = 0; k < K; k++) {
      float t[6];
      for (int j = 0; j < 6; j++) cudaEventElapsedTime(&t[j], tev[0], tev[1 + 6 * k + j]);
      fprintf(stderr, "[tgx] device timeline chunk %llu: H2D %.2f-%.2f  kernels %.2f-%.2f  D2H %.2f-%.2f ms\n",
              (unsigned long long)k, t[0], t[1], t[2], t[3], t[4], t[5]);
    }
    for (auto& e : tev) cudaEventDestroy(e);
  }
  *bad_all_out = bad_all;
  *total = base;
  return TGX_OK;
}

// Input stage of tgx_encode_batch: the H2D copy of a chunk's packed text and its rebased offsets.
struct PackedInput : ChunkInput {
  const uint8_t* text;
  const uint64_t* off;
  std::vector<uint64_t> cut;  // first sample of every chunk
  PackedInput(tgx_model* m, const uint8_t* text_, const uint64_t* off_, uint64_t S) : text(text_), off(off_) {
    const uint64_t N = off[S];
    K = std::max<uint64_t>(1, std::min<uint64_t>(16, (N + m->chunk_bytes - 1) / m->chunk_bytes));
    cut.assign(K + 1, 0);
    cut[K] = S;
    for (uint64_t k = 1; k < K; k++) {
      const uint64_t target = N / K * k;
      uint64_t i = (uint64_t)(std::lower_bound(off, off + S + 1, target) - off);
      cut[k] = std::min<uint64_t>(std::max<uint64_t>(i, cut[k - 1]), S);
    }
    for (uint64_t k = 0; k < K; k++) {
      max_b = std::max(max_b, off[cut[k + 1]] - off[cut[k]]);
      max_s = std::max(max_s, cut[k + 1] - cut[k]);
    }
  }
  int h2d(tgx_model* m, uint64_t k, int b, cudaStream_t st) override {
    const uint64_t s0 = cut[k], s1 = cut[k + 1], b0 = off[s0], nb = off[s1] - b0;
    uint64_t* ho = m->h_off + s0 + k;  // rebased offsets travel through pinned staging (one slice per chunk)
    for (uint64_t i = 0; i <= s1 - s0; i++) ho[i] = off[s0 + i] - b0;
    if (nb) CU(cudaMemcpyAsync(set_text(m, b)->p, text + b0, nb, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(set_off(m, b)->p, ho, (s1 - s0 + 1) * 8, cudaMemcpyHostToDevice, st));
    return TGX_OK;
  }
  int samples(tgx_model*, uint64_t k, int, uint64_t* s0, uint64_t* S, uint64_t* n) override {
    *s0 = cut[k];
    *S = cut[k + 1] - cut[k];
    *n = off[cut[k + 1]] - off[cut[k]];
    return TGX_OK;
  }
};

// Output stage of tgx_encode_batch: u32 ids straight into the caller's buffer, id offsets / status / processed lengths
// through pinned staging (rebased when every chunk is done).
struct PackedOutput : ChunkOutput {
  uint32_t* ids = nullptr;
  uint64_t ids_cap = 0;
  bool want_status = false, want_plen = false;
  uint64_t* st_idoff = nullptr;  // chunk k's S_k + 1 entries at [s0 + k ..]
  int32_t* st_status = nullptr;
  uint64_t* st_plen = nullptr;
  std::vector<uint64_t> bases;
  bool overflow = false;
  int d2h(tgx_model* m, uint64_t k, int b, uint64_t s0, uint64_t Sk, uint64_t tot, uint64_t base, int64_t,
          const int32_t* dst, const uint64_t* dpl, cudaStream_t st) override {
    if (Sk) {
      CU(cudaMemcpyAsync(st_idoff + s0 + k, set_idoff(m, b)->p, (Sk + 1) * 8, cudaMemcpyDeviceToHost, st));
      if (want_status) CU(cudaMemcpyAsync(st_status + s0, dst, Sk * 4, cudaMemcpyDeviceToHost, st));
      if (want_plen) CU(cudaMemcpyAsync(st_plen + s0, dpl, Sk * 8, cudaMemcpyDeviceToHost, st));
    } else {
      st_idoff[s0 + k] = 0;
    }
    if (base + tot > ids_cap) overflow = true;
    if (!overflow && tot) CU(cudaMemcpyAsync(ids + base, set_ids(m, b)->p, tot * 4, cudaMemcpyDeviceToHost, st));
    bases[k] = base;
    return TGX_OK;
  }
};

// Input stage of tgx_encode_corpus: the H2D copy of a raw chunk (cut after a NUL byte) and its split on the device.
// The split's counts are read back through the control stream.  They are queued behind the previous chunk's kernels,
// so the host's wait for them in samples() comes right after its wait for that chunk and overlaps its encode.
struct CorpusInput : ChunkInput {
  const uint8_t* data;
  std::vector<uint64_t> cut;  // first byte of every chunk
  uint64_t next_s0 = 0;       // samples in the chunks split so far
  int64_t bad_sample = -1;    // lowest sample that is not UTF-8 (relative to the buffer), once samples() refused it
  double split_ms = 0;        // device time of the split kernels, all chunks
  CorpusInput(tgx_model* m, const uint8_t* data_, uint64_t n) : data(data_) {
    K = std::max<uint64_t>(1, std::min<uint64_t>(16, (n + m->chunk_bytes - 1) / m->chunk_bytes));
    cut.assign(K + 1, n);
    cut[0] = 0;
    for (uint64_t k = 1; k < K; k++) {  // after the first NUL at or beyond the target: a long sample enlarges its chunk
      const uint64_t from = std::max<uint64_t>(n / K * k, cut[k - 1]);
      const void* z = from < n ? memchr(data + from, 0, n - from) : nullptr;
      cut[k] = z ? (uint64_t)(static_cast<const uint8_t*>(z) - data) + 1 : n;
    }
    for (uint64_t k = 0; k < K; k++) max_b = std::max(max_b, cut[k + 1] - cut[k]);
  }
  int h2d(tgx_model* m, uint64_t k, int b, cudaStream_t st) override {
    const uint64_t nb = cut[k + 1] - cut[k];
    CU(m->raw[b].reserve(max_b + 16));
    if (nb) CU(cudaMemcpyAsync(m->raw[b].p, data + cut[k], nb, cudaMemcpyHostToDevice, st));
    return TGX_OK;
  }
  KeptStarts* tile_counts(tgx_model* m, int b) { return reinterpret_cast<KeptStarts*>(m->split[b].as<unsigned char>() + 32); }
  int after_h2d(tgx_model* m, uint64_t k, int b) override {
    cudaStream_t st = m->w().stream;
    if (K > 1) CU(cudaStreamWaitEvent(st, m->ev_h2d[b], 0));
    const uint64_t N = cut[k + 1] - cut[k], n_tiles = (N + CRLF_TILE - 1) / CRLF_TILE;
    // m->split[b]: bad_pos, words[3], tile counts (n_tiles + 1), their exclusive scan (n_tiles + 1)
    CU(m->split[b].reserve(32 + (n_tiles + 1) * 2 * sizeof(KeptStarts)));
    unsigned long long* bad_pos = m->split[b].as<unsigned long long>();
    unsigned long long* words = bad_pos + 1;
    KeptStarts* cnt = tile_counts(m, b);
    KeptStarts* prefix = cnt + n_tiles + 1;
    CU(cudaEventRecord(m->ev_split[b][0], st));
    CU(dev_fill(bad_pos, 0xFF, 8, st));
    CU(dev_fill(cnt + n_tiles, 0, sizeof(KeptStarts), st));
    const uint8_t* raw = m->raw[b].as<uint8_t>();
    if (n_tiles) corpus_count<<<(uint32_t)n_tiles, CRLF_BLOCK, 0, st>>>(raw, N, cnt, bad_pos);
    size_t tmp = 0;
    CU(cub::DeviceScan::ExclusiveScan(nullptr, tmp, cnt, prefix, AddKeptStarts(), KeptStarts{0, 0}, (int)(n_tiles + 1),
                                      st));
    CU(m->w().cubtmp.reserve(tmp));
    CU(cub::DeviceScan::ExclusiveScan(m->w().cubtmp.p, tmp, cnt, prefix, AddKeptStarts(), KeptStarts{0, 0},
                                      (int)(n_tiles + 1), st));
    corpus_words<<<1, 32, 0, st>>>(raw, prefix, n_tiles, bad_pos, words);
    CU(cudaGetLastError());
    CU(cudaEventRecord(m->ev_split[b][1], st));
    CU(cudaEventRecord(m->w().ev_ctl, st));
    CU(cudaStreamWaitEvent(m->w().stream_ctl, m->w().ev_ctl, 0));
    CU(cudaMemcpyAsync(m->w().h_words + 4, words, 24, cudaMemcpyDeviceToHost, m->w().stream_ctl));
    return TGX_OK;
  }
  int samples(tgx_model* m, uint64_t k, int b, uint64_t* s0, uint64_t* S, uint64_t* n) override {
    CU(cudaStreamSynchronize(m->w().stream_ctl));
    const uint64_t Sk = m->w().h_words[4], kept = m->w().h_words[5], bad = m->w().h_words[6];
    float ms = 0;
    if (cudaEventElapsedTime(&ms, m->ev_split[b][0], m->ev_split[b][1]) == cudaSuccess) split_ms += ms;
    if (bad != ~0ull) {
      bad_sample = (int64_t)(next_s0 + bad);
      return fail(TGX_ERR_NOT_UTF8, "sample " + std::to_string(bad_sample) + " is not valid UTF-8");
    }
    const uint64_t N = cut[k + 1] - cut[k], n_tiles = (N + CRLF_TILE - 1) / CRLF_TILE;
    if (N >= (1ull << 32)) {  // (the kernels index the positions of a sample with 32 bits)
      for (uint64_t p = cut[k]; p < cut[k + 1];) {
        const void* z = memchr(data + p, 0, cut[k + 1] - p);
        const uint64_t e = z ? (uint64_t)(static_cast<const uint8_t*>(z) - data) : cut[k + 1];
        if (e - p >= (1ull << 32)) return fail(TGX_ERR_UNSUPPORTED, "a sample of 4 GiB or more is not supported");
        p = e + 1;
      }
    }
    CU(set_off(m, b)->reserve((Sk + 1) * 8));
    cudaStream_t st = m->w().stream;
    CU(cudaEventRecord(m->ev_split[b][2], st));
    if (n_tiles)
      corpus_scatter<<<(uint32_t)n_tiles, CRLF_BLOCK, 0, st>>>(m->raw[b].as<uint8_t>(), N, tile_counts(m, b) + n_tiles + 1,
                                                               n_tiles, set_text(m, b)->as<uint8_t>(),
                                                               set_off(m, b)->as<uint64_t>());
    CU(cudaGetLastError());
    CU(cudaEventRecord(m->ev_split[b][3], st));
    *s0 = next_s0;
    *S = Sk;
    *n = kept;
    next_s0 += Sk;
    return TGX_OK;
  }
  void add_scatter_ms(tgx_model* m, int b) {  // (chunk's kernels have finished)
    float ms = 0;
    if (cudaEventElapsedTime(&ms, m->ev_split[b][2], m->ev_split[b][3]) == cudaSuccess) split_ms += ms;
  }
};

// Output stage of tgx_encode_corpus: the ids narrowed and separated by corpus_finalize (or the u32 ids as they are)
// and the id offsets straight into the caller's buffers; the offsets are rebased when every chunk is done.
struct CorpusOutput : ChunkOutput {
  CorpusInput* in = nullptr;
  int64_t sep = -1;
  uint32_t id_bytes = 4;
  unsigned char* ids = nullptr;
  uint64_t ids_cap = 0, off_cap = 0;
  uint64_t* id_off = nullptr;
  std::vector<uint64_t> bases, s0s;
  bool ids_overflow = false, off_overflow = false;
  int64_t bad = -1;  // lowest sample without a path (relative to the buffer) and its length after processing
  uint64_t bad_len = 0;
  bool finalize() const { return sep >= 0 || id_bytes == 2; }
  int after_encode(tgx_model* m, uint64_t, int b, uint64_t Sk) override {
    if (!finalize()) return TGX_OK;
    CU(m->fin[b].reserve((in->max_b + 4 + Sk) * id_bytes));
    cudaStream_t st = m->w().stream;
    const uint32_t grid = (uint32_t)m->num_sms * 8;
    const uint32_t* d_ids = set_ids(m, b)->as<uint32_t>();
    const uint64_t* d_idoff = set_idoff(m, b)->as<uint64_t>();
    if (id_bytes == 2)
      corpus_finalize<uint16_t><<<grid, 256, 0, st>>>(d_ids, d_idoff, Sk, sep, m->fin[b].as<uint16_t>());
    else
      corpus_finalize<uint32_t><<<grid, 256, 0, st>>>(d_ids, d_idoff, Sk, sep, m->fin[b].as<uint32_t>());
    m->w().stats.launches += 1;
    CU(cudaGetLastError());
    return TGX_OK;
  }
  int d2h(tgx_model* m, uint64_t k, int b, uint64_t s0, uint64_t Sk, uint64_t tot, uint64_t base, int64_t chunk_bad,
          const int32_t*, const uint64_t* dpl, cudaStream_t st) override {
    if (Sk) in->add_scatter_ms(m, b);  // (the encode that followed the scatter has finished)
    bases[k] = base;
    s0s[k] = s0;
    if (bad < 0 && chunk_bad >= 0) {  // (error path: the length is read at once)
      CU(cudaMemcpyAsync(&bad_len, dpl + chunk_bad, 8, cudaMemcpyDeviceToHost, st));
      CU(cudaStreamSynchronize(st));
      bad = (int64_t)s0 + chunk_bad;
    }
    if (s0 + Sk + 1 > off_cap) off_overflow = true;
    if (!off_overflow && Sk) CU(cudaMemcpyAsync(id_off + s0, set_idoff(m, b)->p, Sk * 8, cudaMemcpyDeviceToHost, st));
    const uint64_t n_out = tot + (sep >= 0 ? Sk : 0), at = base + (sep >= 0 ? s0 : 0);
    if (at + n_out > ids_cap) ids_overflow = true;
    if (!ids_overflow && n_out)
      CU(cudaMemcpyAsync(ids + at * id_bytes, finalize() ? m->fin[b].p : set_ids(m, b)->p, n_out * id_bytes,
                         cudaMemcpyDeviceToHost, st));
    return TGX_OK;
  }
};

}  // namespace

int tgx_encode_batch(tgx_model* m, const uint8_t* text, const uint64_t* off, uint64_t S, uint32_t flags,
                     uint32_t* ids, uint64_t ids_cap, uint64_t* id_off, int32_t* status, uint64_t* proc_len,
                     int64_t* first_bad_out) {
  int rc = check_model(m);
  if (rc) return rc;
  if (!off || !id_off || off[0] != 0) return fail(TGX_ERR_INVALID, "offsets must start at 0");
  for (uint64_t i = 0; i < S; i++) {  // (the reference has no limit on a sample; the kernels index positions with 32 bits)
    if (off[i + 1] < off[i]) return fail(TGX_ERR_INVALID, "offsets must not decrease");
    if (off[i + 1] - off[i] >= (1ull << 32)) return fail(TGX_ERR_UNSUPPORTED, "a sample of 4 GiB or more is not supported");
  }
  std::lock_guard<std::recursive_mutex> g(m->mu);
  struct WiGuard {  // whatever path leaves this function, the next call starts on workspace 0
    tgx_model* m;
    ~WiGuard() { m->wi = 0; }
  } wi_guard{m};
  if (first_bad_out) *first_bad_out = -1;
  if (S == 0) {
    id_off[0] = 0;
    return TGX_OK;
  }
  PackedInput in(m, text, off, S);
  const uint64_t K = in.K;
  // rebased offsets travel through pinned staging (one slice per chunk, alive until the end)
  if (m->h_off_cap < S + K + 1) {
    if (m->h_off) cudaFreeHost(m->h_off);
    m->h_off = nullptr;
    m->h_off_cap = 0;
    CU(cudaHostAlloc(reinterpret_cast<void**>(&m->h_off), (S + K + 1) * 8, cudaHostAllocDefault));
    m->h_off_cap = S + K + 1;
  }
  const uint64_t so_idoff = 0, so_status = (S + K + 1) * 8, so_plen = so_status + ((S * 4 + 15) & ~15ull);
  const uint64_t out_bytes = so_plen + S * 8 + 16;
  if (m->h_out_cap < out_bytes) {
    if (m->h_out) cudaFreeHost(m->h_out);
    m->h_out = nullptr;
    m->h_out_cap = 0;
    CU(cudaHostAlloc(reinterpret_cast<void**>(&m->h_out), out_bytes, cudaHostAllocDefault));
    m->h_out_cap = out_bytes;
  }
  PackedOutput out;
  out.ids = ids;
  out.ids_cap = ids_cap;
  out.want_status = status != nullptr;
  out.want_plen = proc_len != nullptr;
  out.st_idoff = reinterpret_cast<uint64_t*>(m->h_out + so_idoff);
  out.st_status = reinterpret_cast<int32_t*>(m->h_out + so_status);
  out.st_plen = reinterpret_cast<uint64_t*>(m->h_out + so_plen);
  out.bases.assign(K, 0);
  int64_t bad_all = -1;
  uint64_t base = 0;
  rc = encode_chunks(m, flags, 0, in, out, &bad_all, &base);
  if (rc) return rc;
  // chunk-relative id offsets -> global; small outputs leave the pinned staging
  for (uint64_t k = 0; k < K; k++) {
    const uint64_t add = out.bases[k];
    const uint64_t* src = out.st_idoff + in.cut[k] + k;
    for (uint64_t s = in.cut[k]; s < in.cut[k + 1]; s++) id_off[s] = src[s - in.cut[k]] + add;
  }
  id_off[S] = base;
  if (status) std::memcpy(status, out.st_status, S * 4);
  if (proc_len) std::memcpy(proc_len, out.st_plen, S * 8);
  if (first_bad_out) *first_bad_out = bad_all;
  if (out.overflow) return fail(TGX_ERR_CAPACITY, "ids capacity too small: need " + std::to_string(base));
  if (bad_all >= 0) return fail(TGX_ERR_NO_PATH, "no path for sample " + std::to_string(bad_all));
  return TGX_OK;
}

int tgx_encode_corpus(tgx_model* m, const uint8_t* data, uint64_t n, uint32_t flags, uint64_t sample_base,
                      int64_t sep_id, uint32_t id_bytes, void* ids, uint64_t ids_cap, uint64_t* id_off,
                      uint64_t off_cap, uint64_t* n_samples, uint64_t* n_ids, int64_t* first_bad, uint64_t* bad_pos) {
  int rc = check_model(m);
  if (rc) return rc;
  if ((!data && n) || !n_samples || !n_ids || (!ids && ids_cap) || (!id_off && off_cap))
    return fail(TGX_ERR_INVALID, "null argument");
  if (id_bytes != 2 && id_bytes != 4) return fail(TGX_ERR_INVALID, "id_bytes must be 2 or 4");
  if (sep_id < -1 || sep_id >= (int64_t)1 << 32) return fail(TGX_ERR_INVALID, "sep_id must be -1 or a u32 id");
  if (id_bytes == 2 && (m->V > 65536 || sep_id >= 65536))
    return fail(TGX_ERR_UNSUPPORTED, "16-bit ids need a vocabulary (and separator) below 65536");
  std::lock_guard<std::recursive_mutex> g(m->mu);
  struct WiGuard {
    tgx_model* m;
    ~WiGuard() { m->wi = 0; }
  } wi_guard{m};
  *n_samples = *n_ids = 0;
  if (first_bad) *first_bad = -1;
  if (bad_pos) *bad_pos = 0;
  m->last_stats = Stats();
  if (n == 0) {
    if (off_cap < 1) return fail(TGX_ERR_CAPACITY, "offsets capacity too small: need 1");
    id_off[0] = 0;
    return TGX_OK;
  }
  CorpusInput in(m, data, n);
  CorpusOutput out;
  out.in = &in;
  out.sep = sep_id;
  out.id_bytes = id_bytes;
  out.ids = static_cast<unsigned char*>(ids);
  out.ids_cap = ids_cap;
  out.id_off = id_off;
  out.off_cap = off_cap;
  out.bases.assign(in.K, 0);
  out.s0s.assign(in.K, 0);
  int64_t bad_all = -1;
  uint64_t base = 0;
  rc = encode_chunks(m, flags, sample_base, in, out, &bad_all, &base);
  m->last_stats.split_ms = in.split_ms;
  if (rc == TGX_ERR_NOT_UTF8) {  // (lowest invalid sample: the chunks are split in order and stop at the first)
    if (first_bad) *first_bad = in.bad_sample;
    if (bad_pos) {  // byte offset of that sample's first byte: walk the non-empty samples of the buffer
      uint64_t p = 0;
      for (int64_t s = -1;;) {
        while (p < n && data[p] == 0) p++;
        if (++s == in.bad_sample) break;
        const void* z = memchr(data + p, 0, n - p);
        p = z ? (uint64_t)(static_cast<const uint8_t*>(z) - data) : n;
      }
      *bad_pos = p;
    }
    return rc;
  }
  if (rc) return rc;
  const uint64_t S = in.next_s0;
  const uint64_t total = base + (sep_id >= 0 ? S : 0);
  *n_samples = S;
  *n_ids = total;
  if (out.off_overflow || S + 1 > off_cap)
    return fail(TGX_ERR_CAPACITY, "offsets capacity too small: need " + std::to_string(S + 1));
  // chunk-relative id offsets -> global, separators counted
  for (uint64_t k = 0; k < in.K; k++) {
    const uint64_t s0 = out.s0s[k], s1 = k + 1 < in.K ? out.s0s[k + 1] : S;
    for (uint64_t s = s0; s < s1; s++) id_off[s] += out.bases[k] + (sep_id >= 0 ? s : 0);
  }
  id_off[S] = total;
  if (out.ids_overflow) return fail(TGX_ERR_CAPACITY, "ids capacity too small: need " + std::to_string(total));
  if (bad_all >= 0) {
    if (first_bad) *first_bad = bad_all;
    if (bad_pos) *bad_pos = out.bad_len;
    return fail(TGX_ERR_NO_PATH, "no path for sample " + std::to_string(bad_all));
  }
  return TGX_OK;
}

// ---------------------------------------------------------------------------- frequency pass
int tgx_token_frequencies_dev(tgx_model* m, const uint8_t* d_text, const uint64_t* d_off, uint64_t S,
                              uint64_t n_bytes, uint32_t flags, uint64_t* d_freq, int64_t* first_bad_out,
                              uint64_t* bad_len) {
  int rc = check_model(m);
  if (rc) return rc;
  if (!d_off || !d_freq) return fail(TGX_ERR_INVALID, "null argument");
  std::lock_guard<std::recursive_mutex> g(m->mu);
  m->w().stats = Stats();
  cudaStream_t st = m->w().stream;
  if (first_bad_out) *first_bad_out = -1;
  if (S == 0) return TGX_OK;
  CU(cudaEventRecord(m->w().ev[6], st));
  const uint8_t* text = d_text;
  const uint64_t* off = d_off;
  if (flags & TGX_FLAG_CRLF) {
    rc = run_crlf(m, d_text, d_off, S, n_bytes);
    if (rc) return rc;
    text = m->w().text2.as<uint8_t>();
    off = m->w().off2.as<uint64_t>();
  }
  rc = run_viterbi(m, text, off, S, n_bytes, nullptr);
  if (rc) return rc;
  rc = run_emit(m, text, n_bytes, nullptr, 0, reinterpret_cast<unsigned long long*>(d_freq));
  if (rc) return rc;
  int64_t bad = -1;
  rc = first_bad(m, (uint32_t)S, &bad);
  if (rc) return rc;
  CU(cudaEventRecord(m->w().ev[7], st));
  CU(cudaStreamSynchronize(st));
  finish_stats(m, 1);
  if (first_bad_out) *first_bad_out = bad;
  if (bad >= 0) {
    uint32_t l = 0;
    CU(cudaMemcpy(&l, m->w().ulen.as<uint32_t>() + bad, 4, cudaMemcpyDeviceToHost));
    if (bad_len) *bad_len = l;
    return fail(TGX_ERR_NO_PATH, "no path to position " + std::to_string(l) + "/" + std::to_string(l));
  }
  return TGX_OK;
}

int tgx_token_frequencies(tgx_model* m, const uint8_t* text, const uint64_t* off, uint64_t S, uint32_t flags,
                          uint64_t* freq, int64_t* first_bad_out, uint64_t* bad_len) {
  int rc = check_model(m);
  if (rc) return rc;
  if (!off || !freq || off[0] != 0) return fail(TGX_ERR_INVALID, "offsets must start at 0");
  uint64_t N = off[S];
  std::lock_guard<std::recursive_mutex> g(m->mu);
  CU(m->text.reserve(N + 16));
  CU(m->off.reserve((S + 1) * 8));
  CU(m->freq.reserve(m->V * 8 + 8));
  CU(cudaMemcpyAsync(m->text.p, text, N, cudaMemcpyHostToDevice, m->w().stream));
  CU(cudaMemcpyAsync(m->off.p, off, (S + 1) * 8, cudaMemcpyHostToDevice, m->w().stream));
  CU(dev_fill(m->freq.p, 0, m->V * 8 + 8, m->w().stream));
  rc = tgx_token_frequencies_dev(m, m->text.as<uint8_t>(), m->off.as<uint64_t>(), S, N, flags, m->freq.as<uint64_t>(),
                                 first_bad_out, bad_len);
  if (rc) return rc;
  CU(cudaMemcpy(freq, m->freq.p, m->V * 8, cudaMemcpyDeviceToHost));
  return TGX_OK;
}

// ---------------------------------------------------------------------------- pair-frequency pass (merge)
int tgx_pair_frequencies_dev(tgx_model* m, const uint8_t* d_text, const uint64_t* d_off, uint64_t S, uint64_t n_bytes,
                             uint32_t flags, uint64_t* d_pairs, uint64_t* d_counts, uint64_t cap, uint64_t* n_pairs,
                             int64_t* first_bad_out, uint64_t* bad_len) {
  int rc = check_model(m);
  if (rc) return rc;
  if (!d_off || !n_pairs || (cap && (!d_pairs || !d_counts))) return fail(TGX_ERR_INVALID, "null argument");
  std::lock_guard<std::recursive_mutex> g(m->mu);
  *n_pairs = 0;
  if (first_bad_out) *first_bad_out = -1;
  if (S == 0 || n_bytes == 0) return TGX_OK;
  if (S >= (1ull << 32)) return fail(TGX_ERR_INVALID, "too many samples in one call (< 2^32)");
  // 1. encode into the model's own id buffers
  CU(m->ids.reserve((n_bytes + 4) * 4));
  CU(m->idoff.reserve((S + 1) * 8));
  rc = encode_enqueue(m, d_text, d_off, S, n_bytes, flags, m->ids.as<uint32_t>(), n_bytes + 4, m->idoff.as<uint64_t>(),
                      nullptr, nullptr);
  if (rc) return rc;
  uint64_t T = 0;
  int64_t bad = -1;
  rc = encode_finish(m, &T, &bad);
  if (rc) return rc;
  if (bad >= 0) {  // the reference unwraps the encode error (src/merge.rs:59)
    uint32_t l = 0;
    CU(cudaMemcpy(&l, m->w().ulen.as<uint32_t>() + bad, 4, cudaMemcpyDeviceToHost));
    if (first_bad_out) *first_bad_out = bad;
    if (bad_len) *bad_len = l;
    return fail(TGX_ERR_NO_PATH, "no path to position " + std::to_string(l) + "/" + std::to_string(l));
  }
  if (T < 2) return TGX_OK;
  if (T >= (1ull << 31)) return fail(TGX_ERR_INVALID, "too many tokens in one call (< 2^31); split the batch");
  // 2. keys -> sort -> run lengths -> sort by count (stable: ties stay key-ascending)
  cudaStream_t st = m->w().stream;
  const unsigned long long V = std::max<uint64_t>(m->V, 1);
  int key_bits = 1;
  while (key_bits < 64 && (V * V) >> key_bits) key_bits++;
  DevBuf& kb = m->w().bp;      // scratch, free again after the encode: keys | sorted keys
  DevBuf& ub = m->w().mark;    //                                      unique | counts | counts sorted | unique sorted
  DevBuf& nb = m->w().small;
  CU(kb.reserve(T * 16 + 64));
  CU(ub.reserve(T * 32 + 64));
  unsigned long long* keys = kb.as<unsigned long long>();
  unsigned long long* keys_sorted = keys + T;
  unsigned long long* uniq = ub.as<unsigned long long>();
  unsigned long long* cnt = uniq + T;
  unsigned long long* cnt_sorted = cnt + T;
  unsigned long long* uniq_sorted = cnt_sorted + T;
  unsigned long long* d_runs = nb.as<unsigned long long>() + 6;
  unsigned long long* d_np = nb.as<unsigned long long>() + 7;
  pair_keys<<<nblk(T, 256), 256, 0, st>>>(m->ids.as<uint32_t>(), T, V, keys);
  pair_keys_mark_starts<<<nblk(S, 256), 256, 0, st>>>(m->idoff.as<uint64_t>(), S, V, keys);
  size_t tmp = 0;
  CU(cub::DeviceRadixSort::SortKeys(nullptr, tmp, keys, keys_sorted, (int)T, 0, key_bits, st));
  CU(m->w().cubtmp.reserve(tmp));
  CU(cub::DeviceRadixSort::SortKeys(m->w().cubtmp.p, tmp, keys, keys_sorted, (int)T, 0, key_bits, st));
  CU(cub::DeviceRunLengthEncode::Encode(nullptr, tmp, keys_sorted, uniq, cnt, d_runs, (int)T, st));
  CU(m->w().cubtmp.reserve(tmp));
  CU(cub::DeviceRunLengthEncode::Encode(m->w().cubtmp.p, tmp, keys_sorted, uniq, cnt, d_runs, (int)T, st));
  pair_count_runs<<<1, 32, 0, st>>>(uniq, d_runs, V, d_np);
  unsigned long long np = 0;
  rc = read_words(m, d_np, nullptr, &np, nullptr);
  if (rc) return rc;
  *n_pairs = np;
  if (np == 0) return TGX_OK;
  if (np > cap) return fail(TGX_ERR_CAPACITY, "pair capacity too small: need " + std::to_string(np));
  CU(cub::DeviceRadixSort::SortPairsDescending(nullptr, tmp, cnt, cnt_sorted, uniq, uniq_sorted, (int)np, 0, 64, st));
  CU(m->w().cubtmp.reserve(tmp));
  CU(cub::DeviceRadixSort::SortPairsDescending(m->w().cubtmp.p, tmp, cnt, cnt_sorted, uniq, uniq_sorted, (int)np, 0, 64, st));
  pair_unpack<<<nblk(np, 256), 256, 0, st>>>(uniq_sorted, np, V, reinterpret_cast<unsigned long long*>(d_pairs));
  copy_u32<<<nblk(np * 2, 256), 256, 0, st>>>(reinterpret_cast<const uint32_t*>(cnt_sorted),
                                              reinterpret_cast<uint32_t*>(d_counts), np * 2);
  CU(cudaGetLastError());
  CU(cudaStreamSynchronize(st));
  return TGX_OK;
}

int tgx_pair_frequencies(tgx_model* m, const uint8_t* text, const uint64_t* off, uint64_t S, uint32_t flags,
                         uint64_t* pairs, uint64_t* counts, uint64_t cap, uint64_t* n_pairs, int64_t* first_bad_out,
                         uint64_t* bad_len) {
  int rc = check_model(m);
  if (rc) return rc;
  if (!off || !n_pairs || off[0] != 0) return fail(TGX_ERR_INVALID, "offsets must start at 0");
  const uint64_t N = off[S];
  std::lock_guard<std::recursive_mutex> g(m->mu);
  CU(m->text.reserve(N + 16));
  CU(m->off.reserve((S + 1) * 8));
  CU(m->freq.reserve(cap * 16 + 16));
  CU(cudaMemcpyAsync(m->text.p, text, N, cudaMemcpyHostToDevice, m->w().stream));
  CU(cudaMemcpyAsync(m->off.p, off, (S + 1) * 8, cudaMemcpyHostToDevice, m->w().stream));
  uint64_t* d_pairs = m->freq.as<uint64_t>();
  uint64_t* d_counts = d_pairs + cap;
  rc = tgx_pair_frequencies_dev(m, m->text.as<uint8_t>(), m->off.as<uint64_t>(), S, N, flags, d_pairs, d_counts, cap, n_pairs,
                                first_bad_out, bad_len);
  if (rc) return rc;
  if (*n_pairs) {
    CU(cudaMemcpy(pairs, d_pairs, *n_pairs * 8, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(counts, d_counts, *n_pairs * 8, cudaMemcpyDeviceToHost));
  }
  return TGX_OK;
}

// ---------------------------------------------------------------------------- E-step
namespace {

// The E-step over device-resident text.  Results: d_expected[V] += counts (f64) and / or d_limbs[5V] += counts as exact
// integer limbs (tgx_expected_counts_fixed_dev); either may be null.
int expected_counts_impl(tgx_model* m, const uint8_t* d_text, const uint64_t* d_off, uint64_t S, uint64_t n_bytes,
                         uint64_t snippet_len, double* d_expected, long long* d_limbs, int64_t* bad_sample,
                         double* bad_z) {
  int rc = check_model(m);
  if (rc) return rc;
  if (!d_off || (!d_expected && !d_limbs) || snippet_len == 0) return fail(TGX_ERR_INVALID, "bad argument");
  if (snippet_len >= (1ull << 31)) return fail(TGX_ERR_INVALID, "snippet_len must be < 2^31");
  std::lock_guard<std::recursive_mutex> g(m->mu);
  m->w().stats = Stats();
  cudaStream_t st = m->w().stream;
  rc = order_after_caller(m);
  if (rc) return rc;
  CU(cudaEventRecord(m->w().ev[6], st));
  if (bad_sample) *bad_sample = -1;
  if (bad_z) *bad_z = 0.0;
  // 1. snippet table
  CU(m->w().ntok.reserve((S + 2) * 16));
  unsigned long long* cnt = m->w().ntok.as<unsigned long long>();
  unsigned long long* first_unit = cnt + S + 1;
  CU(dev_fill(cnt, 0, (S + 1) * 8, st));
  if (S) {
    snippet_counts<<<nblk(S, 256), 256, 0, st>>>(d_off, S, snippet_len, cnt);
    m->w().stats.launches += 1;
  }
  size_t tmp = 0;
  CU(cub::DeviceScan::ExclusiveSum(nullptr, tmp, cnt, first_unit, (int)(S + 1), st));
  CU(m->w().cubtmp.reserve(tmp));
  CU(cub::DeviceScan::ExclusiveSum(m->w().cubtmp.p, tmp, cnt, first_unit, (int)(S + 1), st));
  m->w().stats.launches += 2;
  unsigned long long U64 = 0;
  CU(cudaMemcpyAsync(&U64, first_unit + S, 8, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  if (U64 >= (1ull << 32)) return fail(TGX_ERR_INVALID, "too many snippets in one call (< 2^32)");
  uint32_t U = (uint32_t)U64;
  if (U == 0) {
    CU(cudaEventRecord(m->w().ev[7], st));
    CU(cudaStreamSynchronize(st));
    return TGX_OK;
  }
  CU(m->w().ustart.reserve((size_t)U * 8 + 8));
  CU(m->w().ulen.reserve((size_t)U * 4 + 4));
  CU(m->w().vals_in.reserve((size_t)U * 4 + 4));
  CU(m->w().status.reserve((size_t)U * 4 + 4));
  CU(m->idoff.reserve((size_t)U * 4 + 4));  // unit -> sample
  CU(m->A.reserve((n_bytes + U + 2) * 8));
  CU(m->w().small.reserve(256));
  units_from_snippets<<<nblk(S, 256), 256, 0, st>>>(d_off, S, snippet_len, first_unit, m->w().ustart.as<uint64_t>(),
                                                   m->w().ulen.as<uint32_t>(), m->w().vals_in.as<uint32_t>(),
                                                   m->idoff.as<uint32_t>());
  m->w().stats.launches += 1;
  rc = sort_units(m, U);
  if (rc) return rc;
  CU(dev_fill(m->w().status.p, 0, (size_t)U * 4 + 4, st));

  FbParams p;
  p.u.text = d_text;
  p.u.unit_start = m->w().ustart.as<uint64_t>();
  p.u.unit_len = m->w().ulen.as<uint32_t>();
  p.u.order = m->w().vals_out.as<uint32_t>();
  p.u.first = 0;
  p.u.count = U;
  p.u.counts = nullptr;
  p.u.part = 0;
  p.u.trie = m->d_trie;
  p.u.root_base = m->da.root_base;
  p.u.rows = std::max<uint32_t>(1, m->da.max_token_len);
  p.u.W = p.u.rows + 1;
  p.A = m->A.as<double>();
  p.status = m->w().status.as<int32_t>();
  p.dropout = m->dropout;
  p.drop_key = drop_unit_key(m->drop_seed, ~0ull);  // (its own stream of draws, apart from the encode samples')
  p.drop_base = m->drop_byte_base;
  p.hot_k = (uint32_t)std::min<uint64_t>(m->V, (uint64_t)m->hot_k);
  p.hot_r = (uint32_t)m->hot_r;
  // fixed-point accumulators of this call (tgx_kernels.cuh: acc_add)
  CU(m->accfix.reserve(m->V * 8 * ACC_LIMBS + 16));
  CU(dev_fill(m->accfix.p, 0, m->V * 8 * ACC_LIMBS + 16, st));
  CU(m->hot.reserve((size_t)p.hot_k * p.hot_r * 8 * ACC_LIMBS + 16));
  CU(dev_fill(m->hot.p, 0, (size_t)p.hot_k * p.hot_r * 8 * ACC_LIMBS, st));
  p.acc = m->accfix.as<unsigned long long>();
  p.hot_acc = m->hot.as<unsigned long long>();
  const bool drop = p.dropout > 0.0;

  // The kernels over the match stream (one lane per snippet; counts from stored alpha / beta) need the match tables
  // and 8 more bytes of device memory per input byte for beta; without them the lane-group kernels take every snippet.
  // Split form (one lane per snippet, beta chains beside the alpha chains, counts from stored alpha / beta): needs 8
  // more bytes of device memory per input byte for beta (+ 4 for the match stream).  Two sets of lane kernels: the ones
  // that walk the trie (fb_split_lane_kernel; faster as measured, profiles/r02_estep_kernels.txt) and the ones over the
  // match stream (fbr_split_kernel; option 19 = 2 selects them).
  // Both take the dropout draw (the walking ones since the end of round 2: 335 against 430 ms per GB at dropout 0.01).
  bool rows_ok = m->estep_split && p.u.rows <= 16;
  if (rows_ok && m->estep_rows == 2) {
    rc = ensure_match_tables(m);
    if (rc) return rc;
  }
  const bool use_rows = rows_ok && m->have_rows && m->estep_rows == 2;
  if (rows_ok) {
    const size_t need = ((size_t)n_bytes + U + 2) * 8 + (use_rows ? ((size_t)n_bytes + 64) * 4 : 0);
    size_t fr = 0, tot = 0;
    const size_t have = m->Bbeta.cap + m->w().rec.cap;
    if (need > have && (cudaMemGetInfo(&fr, &tot) != cudaSuccess || fr + have < need + need / 8 + ((size_t)2 << 30))) rows_ok = false;
    if (rows_ok && m->Bbeta.reserve(((size_t)n_bytes + U + 2) * 8) != cudaSuccess) {
      (void)cudaGetLastError();
      rows_ok = false;
    }
  }
  CU(cudaEventRecord(m->w().ev[8], st));
  if (use_rows) {
    rc = run_match(m, d_text, n_bytes);
    if (rc) return rc;
  }
  CU(cudaEventRecord(m->w().ev[9], st));

  // Long snippets (latency-critical: one ordered chain each) get a whole warp on a second stream; the short ones run
  // one lane each on a third; whatever is in between (only when option 17 sets a lane threshold) G lanes per snippet.
  uint32_t n_long = 0, n_lane = 0;
  {
    uint32_t* counts = m->w().small.as<uint32_t>();
    const bool lanes_ok = rows_ok && m->estep_lane_threshold != 0;
    int64_t thr64 = m->estep_long_threshold;
    if (thr64 <= 0)
      thr64 = (lanes_ok && m->estep_lane_threshold < 0) ? std::max<int64_t>(8192, 16000 + (int64_t)(n_bytes / 30000))
                                                         : std::max<int64_t>(8192, (int64_t)(n_bytes / 18000));
    if (m->g_estep == 32 && !lanes_ok) thr64 = 0x7FFFFFFF;  // one kernel shape for everything
    uint32_t thr = (uint32_t)std::min<int64_t>(thr64, 0x7FFFFFFF);
    uint32_t thr_lane = 0;
    if (lanes_ok)
      thr_lane = m->estep_lane_threshold < 0 ? thr : (uint32_t)std::min<int64_t>(m->estep_lane_threshold, (int64_t)thr);
    split_sorted<<<1, 32, 0, st>>>(m->w().keys_out.as<uint32_t>(), U, thr, thr_lane, counts);
    m->w().stats.launches += 1;
    uint32_t h[3];
    CU(cudaMemcpyAsync(h, counts, 12, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    n_long = h[0];
    n_lane = lanes_ok ? U - h[2] : 0;  // h[2] = units of at least thr_lane bytes
  }
  CU(cudaEventRecord(m->ev_fork, st));
  CU(cudaStreamWaitEvent(m->stream2, m->ev_fork, 0));
  CU(cudaStreamWaitEvent(m->stream3, m->ev_fork, 0));
  FbParams pl = p, ps = p;
  pl.u.first = 0;
  pl.u.count = n_long;
  ps.u.first = n_long;
  ps.u.count = U - n_long - n_lane;
  FbRowsParams pn;
  pn.f = p;
  pn.f.u.first = U - n_lane;
  pn.f.u.count = n_lane;
  pn.rec = m->w().rec.as<uint32_t>();
  pn.rows = m->d_rows.as<double>();
  pn.row_ids = m->d_rowids.as<uint32_t>();
  pn.B = m->Bbeta.as<double>();
  auto contrib_grid = [&](uint32_t units) { return nblk(units, FC_WARPS); };  // a warp per snippet
  FbLaneParams pw;  // the same snippets for the kernels that walk the trie
  pw.f = pn.f;
  pw.blob_end = d_text + n_bytes;
  pw.B = pn.B;
  const bool split = rows_ok;  // beta chains stored and run beside the alpha chains, counts by a third kernel
  const uint32_t lane_blocks = nblk(n_lane, FR_WARPS * 32);
  static_assert(FR_WARPS == FL_WARPS && FRC_WARPS == FC_WARPS, "one launch shape for both sets of lane kernels");
  // forward / backward device times (tgx_model_last_stat 2, 3) are taken on the stream that carries most snippets
  cudaStream_t st_ev = (n_lane > ps.u.count) ? m->stream3 : st;
  (void)st_ev;
  CU(cudaEventRecord(m->w().ev[0], st));  // (tgx_model_last_stat 2 = all chains and counts kernels, 3 = 0)
  CU(launch_fb_g(m, 32, pl, false, m->stream2));
  if (split && pl.u.count) {  // the beta chains of the longest snippets run beside their forward chains
    CU(cudaStreamWaitEvent(m->stream4, m->ev_fork, 0));
    const size_t smem = warp_smem_bytes(pl.u.rows, pl.u.W, 32) * WPB;
    if (drop) {
      CU(cudaFuncSetAttribute(fb_backward_kernel<32, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      fb_backward_kernel<32, true, true><<<nblk(pl.u.count, WPB), WPB * 32, smem, m->stream4>>>(pl, pn.B);
    } else {
      CU(cudaFuncSetAttribute(fb_backward_kernel<32, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      fb_backward_kernel<32, true><<<nblk(pl.u.count, WPB), WPB * 32, smem, m->stream4>>>(pl, pn.B);
    }
    m->w().stats.launches += 1;
    CU(cudaEventRecord(m->ev_join4, m->stream4));
  }
  CU(launch_fb_g(m, m->g_estep, ps, false, st));
  // The lane snippets go in two groups — the longest ones, then the rest — each on a stream of its own: chains, then
  // counts.  The counts kernel is bound by L2 atomics, the chains by instruction issue, so the counts of the first
  // group run beside the chains of the second.  (Measured alternative: four groups whose chain kernels share a stream,
  // the counts on another — 0.90 s against 0.71 s for the 4 GB E-step: every group then waits for the longest chain of
  // the group before it.)
  constexpr int NGRP = 3;
  const double c1 = m->estep_cut1 / 1000.0, c2 = m->estep_cut2 / 1000.0;
  const double grp_cut[NGRP + 1] = {0.0, std::min(c1, c2), c2, 1.0};
  if (n_lane) {
    (void)lane_blocks;
    CU(cudaStreamWaitEvent(m->stream5, m->ev_fork, 0));
    CU(cudaStreamWaitEvent(m->stream6, m->ev_fork, 0));
    for (int gi = 0; gi < NGRP; gi++) {
      const uint32_t g0 = (uint32_t)(n_lane * grp_cut[gi]), g1 = (uint32_t)(n_lane * grp_cut[gi + 1]);
      if (g1 <= g0) continue;
      cudaStream_t gs = gi == 0 ? m->stream3 : (gi == 1 ? m->stream5 : m->stream6);
      FbLaneParams gw = pw;
      gw.f.u.first = pw.f.u.first + g0;
      gw.f.u.count = g1 - g0;
      FbRowsParams gn = pn;
      gn.f.u = gw.f.u;
      const uint32_t blocks = nblk(g1 - g0, FR_WARPS * 32);
      if (!use_rows && drop) fb_split_lane_kernel<true><<<2 * blocks, FL_WARPS * 32, 0, gs>>>(gw);
      else if (!use_rows) fb_split_lane_kernel<false><<<2 * blocks, FL_WARPS * 32, 0, gs>>>(gw);
      else if (drop) fbr_split_kernel<true><<<2 * blocks, FR_WARPS * 32, 0, gs>>>(gn);
      else fbr_split_kernel<false><<<2 * blocks, FR_WARPS * 32, 0, gs>>>(gn);
      if (!use_rows && drop) fb_contrib_kernel<true><<<contrib_grid(g1 - g0), FC_WARPS * 32, 0, gs>>>(gw);
      else if (!use_rows) fb_contrib_kernel<false><<<contrib_grid(g1 - g0), FC_WARPS * 32, 0, gs>>>(gw);
      else if (drop) fbr_contrib_kernel<true><<<contrib_grid(g1 - g0), FRC_WARPS * 32, 0, gs>>>(gn);
      else fbr_contrib_kernel<false><<<contrib_grid(g1 - g0), FRC_WARPS * 32, 0, gs>>>(gn);
      m->w().stats.launches += 2;
    }
  }

  if (split && pl.u.count) {
    CU(cudaStreamWaitEvent(m->stream2, m->ev_join4, 0));
    FbRowsParams pc = pn;
    pc.f.u = pl.u;
    FbLaneParams pcw = pw;
    pcw.f.u = pl.u;
    if (!use_rows && drop) fb_contrib_kernel<true><<<contrib_grid(pl.u.count), FC_WARPS * 32, 0, m->stream2>>>(pcw);
    else if (!use_rows) fb_contrib_kernel<false><<<contrib_grid(pl.u.count), FC_WARPS * 32, 0, m->stream2>>>(pcw);
    else if (drop) fbr_contrib_kernel<true><<<contrib_grid(pl.u.count), FRC_WARPS * 32, 0, m->stream2>>>(pc);
    else fbr_contrib_kernel<false><<<contrib_grid(pl.u.count), FRC_WARPS * 32, 0, m->stream2>>>(pc);
    m->w().stats.launches += 1;
  } else {
    CU(launch_fb_g(m, 32, pl, true, m->stream2));
  }
  CU(launch_fb_g(m, m->g_estep, ps, true, st));
  CU(cudaGetLastError());
  CU(cudaEventRecord(m->ev_join5, m->stream5));
  CU(cudaStreamWaitEvent(st, m->ev_join5, 0));
  CU(cudaEventRecord(m->ev_join6, m->stream6));
  CU(cudaStreamWaitEvent(st, m->ev_join6, 0));
  CU(cudaEventRecord(m->ev_join, m->stream2));
  CU(cudaStreamWaitEvent(st, m->ev_join, 0));
  CU(cudaEventRecord(m->ev_join3, m->stream3));
  CU(cudaStreamWaitEvent(st, m->ev_join3, 0));
  CU(cudaEventRecord(m->w().ev[1], st));
  CU(cudaEventRecord(m->w().ev[2], st));
  CU(cudaEventRecord(m->w().ev[3], st));
  CU(cudaEventRecord(m->ev_join, m->stream2));
  CU(cudaStreamWaitEvent(st, m->ev_join, 0));
  CU(cudaEventRecord(m->ev_join3, m->stream3));
  CU(cudaStreamWaitEvent(st, m->ev_join3, 0));
  fold_hot_acc_kernel<<<nblk(m->V, 256), 256, 0, st>>>(p.hot_acc, p.hot_k, p.hot_r, p.acc, (uint32_t)m->V);
  m->w().stats.launches += 1;
  export_acc_kernel<<<nblk(m->V, 256), 256, 0, st>>>(p.acc, (uint32_t)m->V, d_expected, d_limbs);
  m->w().stats.launches += 1;
  int64_t bad = -1;
  rc = first_bad(m, U, &bad);
  if (rc) return rc;
  CU(cudaEventRecord(m->w().ev[7], st));
  CU(cudaStreamSynchronize(st));
  finish_stats(m, 2);
  float mms = 0;
  if (cudaEventElapsedTime(&mms, m->w().ev[8], m->w().ev[9]) == cudaSuccess) m->last_stats.match_ms = mms;
  if (bad >= 0) {
    uint32_t smp = 0, l = 0;
    uint64_t us = 0;
    CU(cudaMemcpy(&smp, m->idoff.as<uint32_t>() + bad, 4, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(&l, m->w().ulen.as<uint32_t>() + bad, 4, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(&us, m->w().ustart.as<uint64_t>() + bad, 8, cudaMemcpyDeviceToHost));
    double z = 0;
    CU(cudaMemcpy(&z, m->A.as<double>() + us + bad + l, 8, cudaMemcpyDeviceToHost));
    if (bad_sample) *bad_sample = smp;
    if (bad_z) *bad_z = z;
    char buf[160];
    snprintf(buf, sizeof buf, "normalization constant is f64::NaN (z=%g, sample=%u)", z, smp);
    return fail(TGX_ERR_BAD_Z, buf);
  }
  return TGX_OK;
}

}  // namespace

int tgx_expected_counts_dev(tgx_model* m, const uint8_t* d_text, const uint64_t* d_off, uint64_t S,
                            uint64_t n_bytes, uint64_t snippet_len, double* d_expected, int64_t* bad_sample,
                            double* bad_z) {
  if (!d_expected) return fail(TGX_ERR_INVALID, "bad argument");
  return expected_counts_impl(m, d_text, d_off, S, n_bytes, snippet_len, d_expected, nullptr, bad_sample, bad_z);
}

int tgx_expected_counts_fixed_dev(tgx_model* m, const uint8_t* d_text, const uint64_t* d_off, uint64_t S,
                                  uint64_t n_bytes, uint64_t snippet_len, int64_t* d_limbs, int64_t* bad_sample,
                                  double* bad_z) {
  if (!d_limbs) return fail(TGX_ERR_INVALID, "bad argument");
  return expected_counts_impl(m, d_text, d_off, S, n_bytes, snippet_len, nullptr, reinterpret_cast<long long*>(d_limbs),
                              bad_sample, bad_z);
}

int tgx_counts_from_limbs_dev(tgx_model* m, const int64_t* d_limbs, uint64_t vocab_size, double* d_expected) {
  int rc = check_model(m);
  if (rc) return rc;
  if (!d_limbs || !d_expected || vocab_size >= (1ull << 32)) return fail(TGX_ERR_INVALID, "bad argument");
  std::lock_guard<std::recursive_mutex> g(m->mu);
  rc = order_after_caller(m);
  if (rc) return rc;
  if (vocab_size)
    limbs_to_double_kernel<<<nblk(vocab_size, 256), 256, 0, m->w().stream>>>(reinterpret_cast<const long long*>(d_limbs),
                                                                          (uint32_t)vocab_size, d_expected);
  CU(cudaGetLastError());
  CU(cudaStreamSynchronize(m->w().stream));
  return TGX_OK;
}

int tgx_expected_counts(tgx_model* m, const uint8_t* text, const uint64_t* off, uint64_t S,
                        uint64_t snippet_len, double* expected, int64_t* bad_sample, double* bad_z) {
  int rc = check_model(m);
  if (rc) return rc;
  if (!off || !expected || off[0] != 0) return fail(TGX_ERR_INVALID, "offsets must start at 0");
  uint64_t N = off[S];
  std::lock_guard<std::recursive_mutex> g(m->mu);
  CU(m->text.reserve(N + 16));
  CU(m->off.reserve((S + 1) * 8));
  CU(m->expected.reserve(m->V * 8 + 8));
  CU(cudaMemcpyAsync(m->text.p, text, N, cudaMemcpyHostToDevice, m->w().stream));
  CU(cudaMemcpyAsync(m->off.p, off, (S + 1) * 8, cudaMemcpyHostToDevice, m->w().stream));
  CU(dev_fill(m->expected.p, 0, m->V * 8 + 8, m->w().stream));
  rc = tgx_expected_counts_dev(m, m->text.as<uint8_t>(), m->off.as<uint64_t>(), S, N, snippet_len,
                               m->expected.as<double>(), bad_sample, bad_z);
  if (rc) return rc;
  CU(cudaMemcpy(expected, m->expected.p, m->V * 8, cudaMemcpyDeviceToHost));
  return TGX_OK;
}

}  // extern "C"

