// Forward-backward over the match stream: the E-step kernels for snippets that run one per lane (max_token_len <= 16).
//
// Lattice::populate_marginal (src/lattice.rs:245-312) over Model::populate_nodes (src/model.rs:34-55), per-position
// form as in tgx_kernels.cuh (K4/K5): the same folds in the same order, so alpha, beta, z and every contribution are
// bit-identical to the kernels that walk the trie.  What changes is where the matches come from and what a loop trip is:
//   * match_kernel (tgx_match_kernels.cuh) has written, once, the record of every start position; its row
//     (trie_build.h) has a header mask and the scores / ids of the matches dense by length.  The three kernels here
//     read that instead of walking the trie three times.
//   * a trip of the main loop is ONE match per lane: [step to the next position when this one has none left], take the
//     match, log_sum_exp (or exp + accumulate in the counts kernel) — the first term of a fold included, as
//     log_sum_exp(-inf, y), which returns y bit for bit.  (First form of these kernels: a loop of up to four cheap
//     steps per lane in front of the fold; its branches serialised: 10.7 of 32 threads per instruction, 50 ms for the
//     300 MB of profiles/r02_ncu_estep_rows_kernels.txt against 35 ms now.)  In the kernels that probe the trie a
//     trip is one probe and the fold runs only in the lanes whose probe hit a terminal that is not the first of its fold.
//   * populate_nodes' dropout (src/model.rs:48-50) is a keyed draw per (byte offset, length) as in the other E-step
//     kernels, so the three kernels see one lattice.
// Expected counts are accumulated in 128-bit fixed point (64 fraction bits) with integer atomics: the sum does not
// depend on the order of the additions, so counts are bit-identical from run to run, for every chunking of the corpus
// and every number of GPUs (f64 atomics gave a different last bit every run).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "tgx_kernels.cuh"
#include "tgx_match_kernels.cuh"

namespace tgxk {

constexpr int FR_WARPS = 4;

struct FbRowsParams {
  FbParams f;               // units, A, status, accumulators, dropout
  const uint32_t* rec;      // [N] match stream
  const double* rows;       // row table (scores, headers)
  const uint32_t* row_ids;  // row table (ids)
  double* B;                // [N + U] backward log-probabilities (layout of A)
};

// header of the row at `off` (in doubles), cut to the `limit` bytes that are left of the snippet
__device__ __forceinline__ uint32_t fr_mask(double hdr, uint32_t limit) {
  const uint32_t m = (uint32_t)__double_as_longlong(hdr) & 0xFFFFu;
  return limit >= 16u ? m : (m & ((1u << limit) - 1u));
}

template <bool DROP>
__device__ __forceinline__ bool fr_dropped(const FbParams& p, unsigned long long byte_off, uint32_t l) {
  if (!DROP) return false;
  return l > 1u && !(p.dropout < drop_draw(p.drop_key, p.drop_base + byte_off, l));
}

// alpha chains: A[e] = fold over the tokens ending at e, ascending start, of log_sum_exp(., score + A[start]); the
// first term assigns; 0.0 when nothing ends at e (src/lattice.rs:255-272, Q7).
template <bool DROP>
__device__ __forceinline__ void fbr_forward_body(const FbRowsParams& q, uint32_t bid, double* s_win,
                                                 const LibmTabs& lt) {
  const FbParams& p = q.f;
  const UnitParams& u = p.u;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  double* acc = s_win + warp * (16 * 32) + lane;  // slot s at acc[s * 32]
  const uint64_t gidx = (uint64_t)bid * (FR_WARPS * 32) + threadIdx.x;
  const bool has = gidx < u.count;
  const uint32_t unit = has ? u.order[u.first + gidx] : 0;
  const uint32_t n = has ? u.unit_len[unit] : 0;
  const uint64_t start = has ? u.unit_start[unit] : 0;
  double* A = p.A + start + unit;
  const uint32_t* recs = q.rec + start;
  if (has) A[0] = 0.0;
  if (has && n == 0) p.status[unit] = 7;  // z = 0.0 is not normal (Q11)
  bool active = has && n != 0;
  uint32_t pos = 0, seen = 0, m = 0, off = 0;
  // the row of position pos + 1 (offset, header) and the record of position pos + 2 are in flight
  uint32_t noff = 0, rc2 = REC_NOMATCH;
  double nhdr = 0.0;
  if (active) {
    off = (__ldg(recs) & REC_OFF) * 2u;
    m = fr_mask(__ldg(q.rows + off), n);
    if (n > 1) {
      noff = (__ldg(recs + 1) & REC_OFF) * 2u;
      nhdr = __ldg(q.rows + noff);
    }
    if (n > 2) rc2 = __ldg(recs + 2);
  }
  double a = 0.0;  // alpha of the nodes that start at pos
  // A trip = one candidate per lane, and EVERY candidate is a log_sum_exp: the first term of a fold (init_mode,
  // src/lattice.rs:322-323: "return y") goes through the same code with x = -inf — vmax = y > -inf + 50 returns y, the
  // same bits — so a trip has no cheap/expensive lanes: [step to the next position if this one has no match left],
  // take the next match, fold.  (The form with a loop of cheap steps in front of the fold ran 10.7 of 32 threads per
  // instruction: the two branches of that loop serialised, four times per trip.)
  const double ninf = __longlong_as_double(0xFFF0000000000000ll);
  while (__any_sync(0xFFFFFFFFu, active)) {
    // (a position where no token starts — or all of them dropped — takes another trip: rare)
    if (active && !m) {  // everything that ends at pos + 1 has been folded
      pos++;
      const uint32_t sl = pos & 15u;
      a = ((seen >> sl) & 1u) ? acc[sl * 32] : 0.0;
      seen &= ~(1u << sl);
      A[pos] = a;
      if (pos == n) {  // a = alpha[eos]
        const double az = fabs(a);
        const bool normal = (az >= 2.2250738585072014e-308) && (az <= 1.7976931348623157e308);  // f64::is_normal
        p.status[unit] = normal ? 0 : 7;
        active = false;
      } else {
        off = noff;
        m = fr_mask(nhdr, n - pos);
        noff = (rc2 & REC_OFF) * 2u;
        if (pos + 1 < n) nhdr = __ldg(q.rows + noff);
        if (pos + 2 < n) rc2 = __ldg(recs + pos + 2);
      }
    }
    // (measured: letting a lane that met a first term assign it and take a second match in the same trip is slower,
    //  334 against 321 ms per GB: the second take serialises like the old cheap loop)
    bool fold = false;
    uint32_t ts = 0;
    double x = ninf, y = 0.0;
    if (active && m) {
      const uint32_t l = (uint32_t)__ffs((int)m);
      m &= m - 1u;
      if (!fr_dropped<DROP>(p, start + pos, l)) {
        y = __dadd_rn(__ldg(q.rows + off + l), a);  // nodes[lid].score + alpha[lid]
        ts = (pos + l) & 15u;
        if ((seen >> ts) & 1u) x = acc[ts * 32];  // else lid == end_nodes[pos][0]: init_mode
        seen |= 1u << ts;
        fold = true;
      }
    }
    __syncwarp();
    if (fold) acc[ts * 32] = log_sum_exp(x, y, lt);
  }
}

// beta chains: B[p] = fold over the tokens starting at p, ascending length, of log_sum_exp(., score + B[p + len]);
// 0.0 when nothing starts at p (src/lattice.rs:275-287, Q7).  Stored to q.B for fbr_contrib_kernel.
template <bool DROP>
__device__ __forceinline__ void fbr_backward_body(const FbRowsParams& q, uint32_t bid, double* s_win,
                                                  const LibmTabs& lt) {
  const FbParams& p = q.f;
  const UnitParams& u = p.u;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  double* wB = s_win + warp * (16 * 32) + lane;
  const uint64_t gidx = (uint64_t)bid * (FR_WARPS * 32) + threadIdx.x;
  const bool has = gidx < u.count;
  const uint32_t unit = has ? u.order[u.first + gidx] : 0;
  const uint32_t n = has ? u.unit_len[unit] : 0;
  const uint64_t start = has ? u.unit_start[unit] : 0;
  double* Bout = q.B + start + unit;
  const uint32_t* recs = q.rec + start;
  bool active = has && n != 0;
  wB[(n & 15u) * 32] = 0.0;  // beta at the end of the sentence (EOS)
  if (has) Bout[n] = 0.0;
  uint32_t pos = active ? n - 1 : 0, m = 0, off = 0;
  uint32_t noff = 0, rc2 = REC_NOMATCH;
  double nhdr = 0.0;
  if (active) {
    off = (__ldg(recs + pos) & REC_OFF) * 2u;
    m = fr_mask(__ldg(q.rows + off), 1u);
    if (pos >= 1) {
      noff = (__ldg(recs + pos - 1) & REC_OFF) * 2u;
      nhdr = __ldg(q.rows + noff);
    }
    if (pos >= 2) rc2 = __ldg(recs + pos - 2);
  }
  double b = 0.0;  // stays 0.0 when nothing begins at pos (Q7)
  bool first = true;
  const double ninf = __longlong_as_double(0xFFF0000000000000ll);
  while (__any_sync(0xFFFFFFFFu, active)) {  // (trips as in fbr_forward_body)
    if (active && !m) {
      wB[(pos & 15u) * 32] = b;
      Bout[pos] = b;
      if (pos == 0) {
        active = false;
      } else {
        pos--;
        b = 0.0;
        first = true;
        off = noff;
        m = fr_mask(nhdr, n - pos);
        noff = (rc2 & REC_OFF) * 2u;
        if (pos >= 1) nhdr = __ldg(q.rows + noff);
        if (pos >= 2) rc2 = __ldg(recs + pos - 2);
      }
    }
    bool fold = false;
    double x = ninf, y = 0.0;
    if (active && m) {  // ascending length = begin_nodes[pos] order
      const uint32_t l = (uint32_t)__ffs((int)m);
      m &= m - 1u;
      if (!fr_dropped<DROP>(p, start + pos, l)) {
        y = __dadd_rn(__ldg(q.rows + off + l), wB[((pos + l) & 15u) * 32]);  // nodes[rid].score + beta[rid]
        if (!first) x = b;  // else init_mode
        first = false;
        fold = true;
      }
    }
    __syncwarp();
    if (fold) b = log_sum_exp(x, y, lt);
  }
}

// Even blocks run the alpha chains of 128 snippets, odd blocks the beta chains of the same snippets : one
// launch, so that the block scheduler starts the longest snippets of BOTH directions first (two kernels on two streams
// did not interleave: the second kernel's blocks waited for the first kernel's to be dispatched).
template <bool DROP>
__global__ void __launch_bounds__(FR_WARPS * 32) fbr_split_kernel(FbRowsParams q) {
  __shared__ double s_win[FR_WARPS * 16 * 32];
  __shared__ unsigned long long s_et[256];
  __shared__ double s_lt[256];
  const LibmTabs lt = stage_libm_tables(s_et, s_lt);
  if (blockIdx.x & 1u) fbr_backward_body<DROP>(q, blockIdx.x >> 1, s_win, lt);
  else fbr_forward_body<DROP>(q, blockIdx.x >> 1, s_win, lt);
}

// Expected counts from the stored alpha and beta: exp(alpha[pos] + score + beta[pos + len] - z) per matched token, in
// the reference's operation order (src/lattice.rs:295-309).  One warp per snippet, lane i takes the start positions
// i, i + 32, ...; a trip of the main loop is one exp + one accumulation for every lane.
constexpr int FRC_WARPS = 8;

template <bool DROP>
__global__ void __launch_bounds__(FRC_WARPS * 32) fbr_contrib_kernel(FbRowsParams q) {
  __shared__ unsigned long long s_et[256];
  __shared__ double s_lt[256];
  const FbParams& p = q.f;
  const UnitParams& u = p.u;
  const LibmTabs lt = stage_libm_tables(s_et, s_lt);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint64_t widx = (uint64_t)blockIdx.x * FRC_WARPS + warp;
  if (widx >= u.count) return;
  const uint32_t unit = u.order[u.first + widx];
  if (p.status[unit] != 0) return;  // bad z: the reference panics; nothing is added
  const uint32_t n = u.unit_len[unit];
  const uint64_t start = u.unit_start[unit];
  const double* A = p.A + start + unit;
  const double* B = q.B + start + unit;
  const uint32_t* recs = q.rec + start;
  const double z = A[n];
  uint32_t pos = (uint32_t)lane, m = 0, off = 0;
  bool active = pos < n;
  double a = 0.0;
  if (active) {
    off = (__ldg(recs + pos) & REC_OFF) * 2u;
    m = fr_mask(__ldg(q.rows + off), n - pos);
    a = A[pos];
  }
  while (__any_sync(0xFFFFFFFFu, active)) {  // a trip = [next position], one match, one exp + one accumulation per lane
    if (active && !m) {
      pos += 32;
      if (pos >= n) {
        active = false;
      } else {
        off = (__ldg(recs + pos) & REC_OFF) * 2u;
        m = fr_mask(__ldg(q.rows + off), n - pos);
        a = A[pos];
      }
    }
    bool add = false;
    double total = 0.0;
    uint32_t id = 0;
    if (active && m) {
      const uint32_t l = (uint32_t)__ffs((int)m);
      m &= m - 1u;
      if (!fr_dropped<DROP>(p, start + pos, l)) {
        // total = a + score + b - z ; update = total.exp()   (src/lattice.rs:305-307)
        total = __dadd_rn(__dadd_rn(__dadd_rn(a, __ldg(q.rows + off + l)), B[pos + l]), -z);
        id = __ldg(q.row_ids + off + l);
        add = true;
      }
    }
    __syncwarp();
    if (add) acc_add(acc_slot(p, blockIdx.x, id), tgx_exp(total, lt));
  }
}

// replicas of the hot ids -> the accumulators (exact integer sums)
__device__ __host__ __forceinline__ void acc3_add(unsigned long long (&a)[3], const unsigned long long* b) {
  const unsigned long long s0 = a[0] + b[0];
  const unsigned long long c0 = s0 < a[0] ? 1ull : 0ull;
  const unsigned long long s1 = a[1] + b[1];
  unsigned long long c1 = s1 < a[1] ? 1ull : 0ull;
  const unsigned long long s1c = s1 + c0;
  if (s1c < s1) c1++;
  a[0] = s0;
  a[1] = s1c;
  a[2] += b[2] + c1;
}
__global__ void fold_hot_acc_kernel(const unsigned long long* __restrict__ hot_acc, uint32_t hot_k, uint32_t hot_r,
                                    unsigned long long* __restrict__ acc, uint32_t V) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= hot_k || i >= V) return;
  unsigned long long a[3] = {acc[3 * (size_t)i], acc[3 * (size_t)i + 1], acc[3 * (size_t)i + 2]};
  for (uint32_t r = 0; r < hot_r; r++) acc3_add(a, hot_acc + ((size_t)r * hot_k + i) * 3);
  acc[3 * (size_t)i] = a[0];
  acc[3 * (size_t)i + 1] = a[1];
  acc[3 * (size_t)i + 2] = a[2];
}

// accumulators -> the caller's vectors: expected[i] += value (f64), and / or limbs[5i .. 5i+4] += (the four 32-bit
// words of the 128-bit fraction, low to high, and the integer part) — int64 limbs that an integer all-reduce over any
// number of ranks sums exactly (tgx_expected_counts_fixed_dev).
constexpr int COUNT_LIMBS = 5;
// X = ip * 2^128 + f1 * 2^64 + f0  ->  the f64 nearest to X * 2^-128 (ties to even).  X is normalised so that its top
// 64 bits T start with a one; a sticky bit ORed into T's bit 0 stands for the bits below T (bit 0 is far below T's
// rounding position, bit 10), so the one rounding of the u64 -> f64 conversion is the rounding of X itself.  The
// scaling by a power of two is exact: every nonzero X * 2^-128 is at least 2^-128, a normal double.
__device__ __host__ __forceinline__ double fixed_to_double(unsigned long long f0, unsigned long long f1,
                                                           unsigned long long ip) {
  int scale = 128;  // value = (hi * 2^128 + mid * 2^64 + lo) * 2^-scale
  unsigned long long hi = ip, mid = f1, lo = f0;
  if (!hi) { hi = mid; mid = lo; lo = 0; scale += 64; }
  if (!hi) { hi = mid; mid = 0; scale += 64; }
  if (!hi) return 0.0;
#if defined(__CUDA_ARCH__)
  const int s = __clzll((long long)hi);
#else
  const int s = __builtin_clzll(hi);
#endif
  const unsigned long long t = (hi << s) | (s ? mid >> (64 - s) : 0ull);
  const unsigned long long sticky = ((mid << s) | lo) ? 1ull : 0ull;
  // value ~ T * 2^(128 - s - scale); the power of two is built from its exponent field (it is at least 2^-191)
  return (double)(t | sticky) * TGX_AS_F64((unsigned long long)(1023 + 128 - s - scale) << 52);
}
__global__ void export_acc_kernel(const unsigned long long* __restrict__ acc, uint32_t V, double* __restrict__ expected,
                                  long long* __restrict__ limbs) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= V) return;
  const unsigned long long f0 = acc[3 * (size_t)i], f1 = acc[3 * (size_t)i + 1], ip = acc[3 * (size_t)i + 2];
  if (expected) expected[i] += fixed_to_double(f0, f1, ip);
  if (limbs) {
    long long* l = limbs + (size_t)COUNT_LIMBS * i;
    l[0] += (long long)(f0 & 0xFFFFFFFFull);
    l[1] += (long long)(f0 >> 32);
    l[2] += (long long)(f1 & 0xFFFFFFFFull);
    l[3] += (long long)(f1 >> 32);
    l[4] += (long long)ip;
  }
}
// limbs (after any number of exact integer sums) -> f64
__global__ void limbs_to_double_kernel(const long long* __restrict__ limbs, uint32_t V, double* __restrict__ expected) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= V) return;
  const long long* l = limbs + (size_t)COUNT_LIMBS * i;
  unsigned long long w[4], ip = (unsigned long long)l[4], carry = 0;
#pragma unroll
  for (int k = 0; k < 4; k++) {
    const unsigned long long v = (unsigned long long)l[k] + carry;
    w[k] = v & 0xFFFFFFFFull;
    carry = v >> 32;
  }
  ip += carry;
  expected[i] = fixed_to_double((w[1] << 32) | w[0], (w[3] << 32) | w[2], ip);
}

}  // namespace tgxk
