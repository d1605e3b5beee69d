// =============================================================================
// oracle/tgx_oracle.cpp — CPU restatement of the TokenGeeX hot path.
//
// TEST INFRASTRUCTURE ONLY.  Nothing under tokengeex_b200/ (the product) links,
// imports or executes this file.  Only tests/, __graft_entry__.smoke() and
// bench.py's cpu_baseline / `--impl reference` legs may load liboracle.so.
//
// The reference (rojas-diego/tokengeex) is pure Rust and there is no Rust
// toolchain in this image, so the reference itself cannot be compiled here
// (oracle/_ref does not exist).  This file restates its algorithms function by
// function in C++17, keeping the reference's data structures (pointer trie with
// a per-node byte-keyed FNV hash map, 32-byte dp nodes, node-arena lattice with
// begin/end adjacency) and its evaluation order, so results are the
// reference's bit for bit wherever the reference itself is deterministic.
// Compile with -O2 -ffp-contract=off (Rust never contracts a*b+c into an FMA);
// exp/ln go to the platform libm exactly as Rust's f64::exp / f64::ln do.
//
// Pinning: the reference's own tests hold goldens for Model::encode
// (src/model.rs:209-252), the special-token splitter (src/tokenizer.rs:442-486)
// and - commented out - forward-backward marginals (src/lattice.rs:417-452).
// tests/test_oracle_goldens.py checks all of them.  run_e_step / run_m_step /
// prune_vocab / nbest have NO golden in the reference ("parity unpinned" by the
// reference's tests); they are pinned here by line-by-line restatement plus an
// independent brute-force path enumerator (tests/bruteforce.py (used by tests/test_oracle_goldens.py)).
//
// Every function cites the reference file:line it follows (paths relative to
// /root/reference).
// =============================================================================
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <limits>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

namespace orc {

// ----------------------------------------------------------------------------
// src/lib.rs:19-31  TokenID = u32, ScoredToken { value, score, keep }
// ----------------------------------------------------------------------------
struct ScoredToken {
  std::vector<uint8_t> value;
  double score;
  bool keep;
};

// ----------------------------------------------------------------------------
// src/trie.rs:75-78  Node { data: Option<Data>, children: HashMap<u8,Node,Fnv> }
// Restated as an arena of nodes; every node owns a small open-addressing table
// keyed by the edge byte and hashed with FNV-1a (the fnv crate's hasher), which
// is what `HashMap<u8, Node, FnvBuildHasher>` amounts to.
// ----------------------------------------------------------------------------
struct TrieNode {
  bool has_data = false;
  uint32_t id = 0;    // Data = (TokenID, u32 len)   src/model.rs:12
  uint32_t len = 0;
  // open addressing table: slots hold (key+1) in `keys` (0 = empty)
  std::vector<uint16_t> keys;
  std::vector<uint32_t> vals;
  uint32_t count = 0;
};

static inline uint64_t fnv1a_u8(uint8_t b) {
  uint64_t h = 0xcbf29ce484222325ULL;
  h ^= b;
  h *= 0x100000001b3ULL;
  return h;
}

struct Trie {
  std::vector<TrieNode> nodes;
  Trie() { nodes.emplace_back(); }

  int32_t child(uint32_t n, uint8_t b) const {
    const TrieNode& nd = nodes[n];
    if (nd.keys.empty()) return -1;
    size_t mask = nd.keys.size() - 1;
    size_t i = (size_t)(fnv1a_u8(b) >> 7) & mask;
    for (;;) {
      uint16_t k = nd.keys[i];
      if (k == 0) return -1;
      if (k == (uint16_t)b + 1) return (int32_t)nd.vals[i];
      i = (i + 1) & mask;
    }
  }

  void grow(uint32_t n) {
    TrieNode& nd = nodes[n];
    size_t ncap = nd.keys.empty() ? 4 : nd.keys.size() * 2;
    std::vector<uint16_t> ok;
    std::vector<uint32_t> ov;
    ok.swap(nd.keys);
    ov.swap(nd.vals);
    nd.keys.assign(ncap, 0);
    nd.vals.assign(ncap, 0);
    size_t mask = ncap - 1;
    for (size_t j = 0; j < ok.size(); j++) {
      if (!ok[j]) continue;
      size_t i = (size_t)(fnv1a_u8((uint8_t)(ok[j] - 1)) >> 7) & mask;
      while (nd.keys[i]) i = (i + 1) & mask;
      nd.keys[i] = ok[j];
      nd.vals[i] = ov[j];
    }
  }

  uint32_t child_or_insert(uint32_t n, uint8_t b) {
    int32_t c = child(n, b);
    if (c >= 0) return (uint32_t)c;
    if (nodes[n].keys.empty() || (nodes[n].count + 1) * 4 > nodes[n].keys.size() * 3) grow(n);
    uint32_t nn = (uint32_t)nodes.size();
    nodes.emplace_back();
    TrieNode& nd = nodes[n];
    size_t mask = nd.keys.size() - 1;
    size_t i = (size_t)(fnv1a_u8(b) >> 7) & mask;
    while (nd.keys[i]) i = (i + 1) & mask;
    nd.keys[i] = (uint16_t)b + 1;
    nd.vals[i] = nn;
    nd.count++;
    return nn;
  }

  // src/trie.rs:12-20  Trie::push — walks/creates one child per byte, then
  // overwrites node.data (so a duplicate byte string keeps the LAST data).
  void push(const uint8_t* e, size_t n, uint32_t id, uint32_t len) {
    uint32_t node = 0;
    for (size_t i = 0; i < n; i++) node = child_or_insert(node, e[i]);
    nodes[node].has_data = true;
    nodes[node].id = id;
    nodes[node].len = len;
  }
};

// src/trie.rs:38-63  TrieIterator: consume one byte, step to the child (stop at
// the first missing edge), yield node.data when present.  `f(id,len)` is called
// for every yielded item, in increasing length.
template <class F>
static inline void common_prefix_search(const Trie& t, const uint8_t* s, size_t n, F&& f) {
  uint32_t node = 0;
  for (size_t i = 0; i < n; i++) {
    int32_t c = t.child(node, s[i]);
    if (c < 0) return;
    node = (uint32_t)c;
    const TrieNode& nd = t.nodes[node];
    if (nd.has_data) f(nd.id, nd.len);
  }
}

// ----------------------------------------------------------------------------
// src/model.rs:8-30  Model { vocab, token_to_ids, trie } and Model::from
// ----------------------------------------------------------------------------
struct Model {
  std::vector<ScoredToken> vocab;
  Trie trie;
  uint64_t rng_state = 0x9E3779B97F4A7C15ULL;  // dropout>0 only (see encode)

  explicit Model(std::vector<ScoredToken> v) : vocab(std::move(v)) {
    for (size_t id = 0; id < vocab.size(); id++)
      trie.push(vocab[id].value.data(), vocab[id].value.size(), (uint32_t)id,
                (uint32_t)vocab[id].value.size());
  }
  size_t vocab_size() const { return vocab.size(); }
};

// splitmix64 → uniform [0,1).  The reference uses rand::random::<f64>()
// (unseeded thread_rng, src/model.rs:48,100) — not reproducible by anyone, so
// for 0 < dropout < 1 only the distribution can agree.  dropout <= 0 and
// dropout >= 1 never depend on the draw's value and are exact.
static inline double next_f64(uint64_t& s) {
  uint64_t z = (s += 0x9E3779B97F4A7C15ULL);
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
  z ^= z >> 31;
  return (double)(z >> 11) * (1.0 / 9007199254740992.0);
}

// Keyed draw for dropout parity tests: the product's documented stand-in for rand::random::<f64>()
// (include/tokengeex_b200.h, tgx_model_set_dropout) restated — a pure function of (seed, sample index,
// start position, token length): two rounds of the splitmix64 finaliser, 53-bit uniform in [0,1).
static inline uint64_t drop_mix(uint64_t z) {
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
  return z ^ (z >> 31);
}
struct KeyedDraw {
  uint64_t unit_key;
  KeyedDraw(uint64_t seed, uint64_t sample) : unit_key(drop_mix(seed + 0x9E3779B97F4A7C15ULL * (sample + 1))) {}
  double operator()(uint64_t pos, uint32_t len) const {
    uint64_t z = drop_mix(unit_key + 0x9E3779B97F4A7C15ULL * ((pos << 8) | len));
    return (double)(z >> 11) * (1.0 / 9007199254740992.0);
  }
};

// ----------------------------------------------------------------------------
// src/model.rs:59-129  Model::encode  (Viterbi, "SentencePiece DP")
// Returns 0 on success; 1 = Error::NoPath(pos,len) (src/lib.rs:243-245).
// ----------------------------------------------------------------------------
struct DpNode {  // src/model.rs:63-68  struct Node { id, score, start: Option<usize> }
  uint32_t id;
  double score;
  uint64_t start;
  bool has_start;
};

static int encode(const Model& m, const uint8_t* input, size_t n, double dropout,
                  std::vector<uint32_t>& ids, uint64_t* err_pos, uint64_t* err_len,
                  uint64_t* rng, const KeyedDraw* keyed = nullptr) {
  ids.clear();
  std::vector<DpNode> dp(n + 1, DpNode{0, 0.0, 0, false});  // :72-79
  dp[0].has_start = true;                                   // :81  dp[0].start = Some(0)
  dp[0].start = 0;

  for (size_t pos = 0; pos < n; pos++) {  // :83
    if (!dp[pos].has_start) continue;     // :85-87 unreachable positions are skipped
    common_prefix_search(m.trie, input + pos, n - pos, [&](uint32_t id, uint32_t len32) {  // :92-95
      size_t len = len32;
      const DpNode& node = dp[pos + len];                      // :96-97
      double score = dp[pos].score + m.vocab[id].score;        // :98
      // :100  (dropout <= 0.0 || len <= 1 || dropout < rand::random::<f64>())
      //       && (node.start.is_none() || score > node.score)
      bool keep = dropout <= 0.0 || len <= 1;
      if (!keep) keep = dropout < (keyed ? (*keyed)(pos, len32) : next_f64(*rng));
      if (keep && (!node.has_start || score > node.score)) {
        dp[pos + len] = DpNode{id, score, pos, true};          // :103-107
      }
    });
  }

  // :113-123 backtrack
  size_t pos = n;
  ids.reserve(n / 2);
  while (pos > 0) {
    const DpNode& node = dp[pos];
    if (!node.has_start) {  // :119  ok_or_else(|| Error::NoPath(pos, input.len()))
      *err_pos = pos;
      *err_len = n;
      ids.clear();
      return 1;
    }
    ids.push_back(node.id);
    pos = node.start;
  }
  std::reverse(ids.begin(), ids.end());  // :126
  return 0;
}

// ----------------------------------------------------------------------------
// src/processor.rs:47-49  CrlfProcessor::preprocess = s.replace("\r\n", "\n")
// (Rust str::replace: non-overlapping matches, left to right.)
// ----------------------------------------------------------------------------
static size_t crlf(const uint8_t* s, size_t n, uint8_t* out) {
  size_t o = 0;
  size_t i = 0;
  while (i < n) {
    if (s[i] == '\r' && i + 1 < n && s[i + 1] == '\n') {
      out[o++] = '\n';
      i += 2;
    } else {
      out[o++] = s[i++];
    }
  }
  return o;
}

// ----------------------------------------------------------------------------
// src/lattice.rs:13-26  Node   /  :51-65 Lattice
// ----------------------------------------------------------------------------
struct LNode {
  size_t pos;
  uint32_t token_id;
  size_t token_len;
  double score;
  int64_t prev;  // Option<usize>: -1 = None
  double backtrack_score;
};

struct Lattice {
  const uint8_t* sentence = nullptr;
  size_t len = 0;
  std::vector<std::vector<size_t>> begin_nodes, end_nodes;
  std::vector<LNode> nodes;
  size_t bos_idx = 0, eos_idx = 0;

  // src/lattice.rs:78-103  Lattice::from
  void from(const uint8_t* s, size_t n) {
    sentence = s;
    len = n;
    nodes.clear();
    begin_nodes.assign(n + 1, {});
    end_nodes.assign(n + 1, {});
    nodes.push_back(LNode{0, 0xFFFFFFFEu, 0, 0.0, -1, 0.0});  // BOS = TokenID::MAX-1  :96
    bos_idx = 0;
    nodes.push_back(LNode{n, 0xFFFFFFFFu, 0, 0.0, -1, 0.0});  // EOS = TokenID::MAX    :98-99
    eos_idx = 1;
    end_nodes[0].push_back(bos_idx);    // :101
    begin_nodes[n].push_back(eos_idx);  // :102
  }

  // src/lattice.rs:105-110  Lattice::insert
  void insert(size_t pos, uint32_t id, size_t tlen, double score) {
    size_t idx = nodes.size();
    begin_nodes[pos].push_back(idx);
    end_nodes[pos + tlen].push_back(idx);
    nodes.push_back(LNode{pos, id, tlen, score, -1, 0.0});
  }

  // src/lattice.rs:112-150  Lattice::viterbi — returns node indices (path
  // includes EOS, excludes BOS: every node whose prev is Some, from EOS back).
  std::vector<size_t> viterbi() {
    for (size_t pos = 0; pos <= len; pos++) {
      for (size_t rnode : begin_nodes[pos]) {
        nodes[rnode].prev = -1;
        double best_score = 0.0;
        int64_t best_node = -1;
        for (size_t lnode : end_nodes[pos]) {
          double score = nodes[lnode].backtrack_score + nodes[rnode].score;
          if (best_node < 0 || score > best_score) {
            best_node = (int64_t)lnode;
            best_score = score;
          }
        }
        if (best_node < 0) return {};  // :131-133
        nodes[rnode].prev = best_node;
        nodes[rnode].backtrack_score = best_score;
      }
    }
    std::vector<size_t> results;
    size_t node_idx = begin_nodes[len][0];
    while (nodes[node_idx].prev >= 0) {  // :142-146
      results.push_back(node_idx);
      node_idx = (size_t)nodes[node_idx].prev;
    }
    std::reverse(results.begin(), results.end());
    return results;
  }
};

// src/model.rs:34-55  Model::populate_nodes (dropout restated with the same
// caveat as encode; every position is walked, reachable or not).
// `keyed`: the product's keyed draw (tgx_model_set_dropout) instead of the sequential one; position = pos_base + pos.
// The reference drops when `rand < dropout`; the keyed rule is the encode rule, keep iff `dropout < u` (the two
// differ only on the null event u == dropout).
static void populate_nodes(const Model& m, Lattice& lat, double dropout, uint64_t* rng,
                           const KeyedDraw* keyed = nullptr, uint64_t pos_base = 0) {
  for (size_t pos = 0; pos < lat.len; pos++) {
    common_prefix_search(m.trie, lat.sentence + pos, lat.len - pos, [&](uint32_t id, uint32_t len) {
      double score = m.vocab[id].score;
      if (len > 1 && dropout > 0.0 &&
          (keyed ? !(dropout < (*keyed)(pos_base + pos, len)) : next_f64(*rng) < dropout)) return;  // :48-50
      lat.insert(pos, id, len, score);                                  // :52
    });
  }
}

// src/lattice.rs:321-333  log_sum_exp
static inline double log_sum_exp(double x, double y, bool init_mode) {
  if (init_mode) return y;
  double vmin, vmax;
  if (x > y) { vmin = y; vmax = x; } else { vmin = x; vmax = y; }
  const double k_minus_log_epsilon = 50.0;
  if (vmax > vmin + k_minus_log_epsilon) return vmax;
  return vmax + std::log(std::exp(vmin - vmax) + 1.0);
}

// Exact fixed-point sums of the contributions (tests only): fixed[3 * id + 0 / 1 / 2] = bits 65..128 / bits 1..64 /
// integer part of sum(floor(c * 2^128)) mod 2^192, a 192-bit integer kept as three u64 words (low to high).  The floor
// is derived from c's significand and exponent, independently of the product's decomposition (acc_add).  The modulus
// only matters for a contribution of 2^64 or more, which the product's accumulators cannot hold either; only a lattice
// with positions nothing begins at (beta = log 1 there, src/lattice.rs:275-287) can produce one.
static inline void fixed_merge(uint64_t* w, const uint64_t* x) {  // w += x (mod 2^192)
  uint64_t carry = 0;
  for (int k = 0; k < 3; k++) {
    const unsigned __int128 t = (unsigned __int128)w[k] + x[k] + carry;
    w[k] = (uint64_t)t;
    carry = (uint64_t)(t >> 64);
  }
}
static inline void fixed_add(uint64_t* w, double c) {
  if (!(c > 0.0) || !std::isfinite(c)) return;  // exp() >= 0; a NaN only comes from a bad z (reported as such)
  int e = 0;
  const double f = std::frexp(c, &e);  // c = f * 2^e, f in [0.5, 1)
  const uint64_t m = (uint64_t)std::ldexp(f, 53);  // exact: c = m * 2^(e - 53), m < 2^53
  const int s = e - 53 + 128;  // c * 2^128 = m * 2^s
  uint64_t add[3] = {0, 0, 0};
  if (s < 0) {
    if (s > -64) add[0] = m >> -s;  // the floor: the bits shifted out are dropped
  } else {
    const int wi = s / 64, b = s % 64;
    if (wi < 3) add[wi] = m << b;
    if (b && wi + 1 < 3) add[wi + 1] = m >> (64 - b);
  }
  fixed_merge(w, add);
}

// Optional outputs of the marginal functions beside expected[]: the exact fixed-point sums and / or the list of
// (id, contribution) in the order they are added.
struct MarginalSinks {
  uint64_t* fixed = nullptr;                             // [V][3]
  std::vector<std::pair<uint32_t, double>>* contribs = nullptr;
  void add(uint32_t id, double c) const {
    if (fixed) fixed_add(fixed + 3 * (size_t)id, c);
    if (contribs) contribs->emplace_back(id, c);
  }
};

// src/lattice.rs:245-312  Lattice::populate_marginal — literal restatement,
// including the O(|begin|*|end|) double loops.
static double populate_marginal(const Lattice& lat, double* expected, const MarginalSinks* sinks = nullptr) {
  size_t len = lat.len;
  size_t num_nodes = lat.nodes.size();
  std::vector<double> alpha(num_nodes, 0.0), beta(num_nodes, 0.0);
  for (size_t pos = 0; pos <= len; pos++) {  // :259-272
    for (size_t rid : lat.begin_nodes[pos]) {
      for (size_t lid : lat.end_nodes[pos]) {
        alpha[rid] = log_sum_exp(alpha[rid], lat.nodes[lid].score + alpha[lid],
                                 lid == lat.end_nodes[pos][0]);
      }
    }
  }
  for (size_t pos = len + 1; pos-- > 0;) {  // :275-287
    for (size_t lid : lat.end_nodes[pos]) {
      for (size_t rid : lat.begin_nodes[pos]) {
        beta[lid] = log_sum_exp(beta[lid], lat.nodes[rid].score + beta[rid],
                                rid == lat.begin_nodes[pos][0]);
      }
    }
  }
  double z = alpha[lat.eos_idx];  // :290-291
  for (size_t pos = 0; pos < len; pos++) {  // :295-309
    for (size_t node_idx : lat.begin_nodes[pos]) {
      uint32_t id = lat.nodes[node_idx].token_id;
      double score = lat.nodes[node_idx].score;
      double a = alpha[node_idx];
      double b = beta[node_idx];
      double total = a + score + b - z;
      double update = std::exp(total);
      expected[id] += update;
      if (sinks) sinks->add(id, update);
    }
  }
  return z;
}

// Per-position form of the same computation (SURVEY.md §8 a7): every right node
// at `pos` performs the identical fold over end_nodes[pos], so alpha depends on
// pos only (A[pos]); likewise beta depends on the node's end position (B[pos]).
// Same operations in the same order ⇒ bit-identical to populate_marginal; this
// is what the CPU baseline times and what the CUDA kernels restate.
static double marginal_per_position(const Model& m, const uint8_t* s, size_t n, double* expected,
                                    std::vector<double>& A, std::vector<double>& B,
                                    std::vector<uint8_t>& seen, const MarginalSinks* sinks = nullptr) {
  A.assign(n + 1, 0.0);
  B.assign(n + 1, 0.0);
  seen.assign(n + 1, 0);
  // forward, push form: contributions to A[e] arrive in ascending start order,
  // which is end_nodes[e]'s order (nodes are inserted by pos asc, len asc).
  // A[0] = log_sum_exp(0, BOS.score + alpha[BOS], init) = 0.0 + 0.0.
  A[0] = 0.0 + 0.0;
  seen[0] = 1;
  for (size_t pos = 0; pos < n; pos++) {
    double a = A[pos];  // final: all starts < pos have pushed
    common_prefix_search(m.trie, s + pos, n - pos, [&](uint32_t id, uint32_t len) {
      double y = m.vocab[id].score + a;
      size_t e = pos + len;
      A[e] = log_sum_exp(A[e], y, !seen[e]);
      seen[e] = 1;
    });
  }
  double z = A[n];
  // backward, pull form: begin_nodes[pos] is in ascending length order.
  // B[n] = log_sum_exp(0, EOS.score + beta[EOS], init) = 0.0 + 0.0.
  B[n] = 0.0 + 0.0;
  for (size_t pos = n; pos-- > 0;) {
    bool first = true;
    double b = 0.0;  // stays 0.0 when nothing begins at pos  (Q7)
    common_prefix_search(m.trie, s + pos, n - pos, [&](uint32_t id, uint32_t len) {
      b = log_sum_exp(b, m.vocab[id].score + B[pos + len], first);
      first = false;
    });
    B[pos] = b;
  }
  // expected counts, positions ascending / lengths ascending — the same
  // accumulation order as src/lattice.rs:295-309, so the sums round identically.
  for (size_t pos = 0; pos < n; pos++) {
    double a = A[pos];
    common_prefix_search(m.trie, s + pos, n - pos, [&](uint32_t id, uint32_t len) {
      double sc = m.vocab[id].score;
      double total = a + sc + B[pos + len] - z;
      const double update = std::exp(total);
      expected[id] += update;
      if (sinks) sinks->add(id, update);
    });
  }
  return z;
}

// ----------------------------------------------------------------------------
// src/lattice.rs:336-378  Hypothesis + Agenda (Rust std BinaryHeap restated:
// SURVEY.md Appendix D).  cmp: Less iff self.fx < other.fx else Greater.
// `a <= b` ⇔ a.fx < b.fx.
// ----------------------------------------------------------------------------
struct Hyp {
  size_t node_idx;
  int64_t next;  // index into hyp arena, -1 = None
  double fx, gx;
};

struct Agenda {
  std::vector<int64_t> data;  // indices into arena
  const std::vector<Hyp>* arena = nullptr;
  bool le(int64_t a, int64_t b) const { return (*arena)[a].fx < (*arena)[b].fx; }
  size_t size() const { return data.size(); }
  void sift_up(size_t start, size_t pos) {
    int64_t elem = data[pos];
    while (pos > start) {
      size_t parent = (pos - 1) / 2;
      if (le(elem, data[parent])) break;
      data[pos] = data[parent];
      pos = parent;
    }
    data[pos] = elem;
  }
  void push(int64_t h) {
    data.push_back(h);
    sift_up(0, data.size() - 1);
  }
  void sift_down_to_bottom(size_t pos) {
    size_t end = data.size();
    size_t start = pos;
    int64_t elem = data[pos];
    size_t child = 2 * pos + 1;
    while (child + 1 < end) {  // child <= end.saturating_sub(2)
      if (le(data[child], data[child + 1])) child += 1;
      data[pos] = data[child];
      pos = child;
      child = 2 * pos + 1;
    }
    if (child == end - 1) {
      data[pos] = data[child];
      pos = child;
    }
    data[pos] = elem;
    sift_up(start, pos);
  }
  int64_t pop() {
    int64_t item = data.back();
    data.pop_back();
    if (!data.empty()) {
      std::swap(item, data[0]);
      sift_down_to_bottom(0);
    }
    return item;
  }
};

// src/lattice.rs:152-238  Lattice::nbest — returns paths as node-index lists.
static std::vector<std::vector<size_t>> nbest(Lattice& lat, size_t n) {
  std::vector<std::vector<size_t>> hypotheses;
  if (n == 0) return hypotheses;
  if (n == 1) {
    hypotheses.push_back(lat.viterbi());
    return hypotheses;
  }
  std::vector<Hyp> arena;
  Agenda agenda;
  agenda.arena = &arena;
  size_t eos_id = 1;
  double score = lat.nodes[eos_id].score;
  arena.push_back(Hyp{eos_id, -1, score, score});
  agenda.push(0);
  lat.viterbi();
  while (agenda.size() > 0) {
    int64_t top = agenda.pop();
    size_t node_idx = arena[top].node_idx;
    uint32_t node_id = lat.nodes[node_idx].token_id;
    uint32_t bos_node_id = lat.nodes[lat.bos_idx].token_id;
    size_t node_pos = lat.nodes[node_idx].pos;
    if (node_id == bos_node_id) {  // :179
      std::vector<size_t> hypothesis;
      int64_t next = arena[top].next;
      while (arena[next].next >= 0) {  // :184-190
        hypothesis.push_back(arena[next].node_idx);
        next = arena[next].next;
      }
      hypotheses.push_back(hypothesis);
      if (hypotheses.size() == n) return hypotheses;
    } else {
      for (size_t lnode : lat.end_nodes[node_pos]) {  // :201-207
        double top_gx = arena[top].gx;
        double fx = lat.nodes[lnode].backtrack_score + top_gx;
        double gx = lat.nodes[lnode].score + top_gx;
        arena.push_back(Hyp{lnode, top, fx, gx});
        agenda.push((int64_t)arena.size() - 1);
      }
      const size_t k_max_agenda_size = 100000, k_min_agenda_size = 512;  // :211-228
      if (agenda.size() > k_max_agenda_size) {
        Agenda na;
        na.arena = &arena;
        size_t l = std::min(k_min_agenda_size, n * 10);
        for (size_t i = 0; i < l; i++) na.push(agenda.pop());
        agenda.data.swap(na.data);
      }
    }
  }
  return hypotheses;
}

// ----------------------------------------------------------------------------
// src/task.rs:134-137  par_chunk_size
// ----------------------------------------------------------------------------
static size_t par_chunk_size(size_t num_samples, size_t threads, size_t f) {
  size_t c = num_samples / threads / f;
  return std::max<size_t>(1, c);
}

template <class F>
static void parallel_chunks(size_t n_items, size_t chunk, int threads, F&& f) {
  size_t n_chunks = (n_items + chunk - 1) / chunk;
  std::atomic<size_t> next{0};
  auto worker = [&](int tid) {
    for (;;) {
      size_t c = next.fetch_add(1);
      if (c >= n_chunks) break;
      f(c, c * chunk, std::min(n_items, (c + 1) * chunk), tid);
    }
  };
  if (threads <= 1) { worker(0); return; }
  std::vector<std::thread> ts;
  for (int t = 0; t < threads; t++) ts.emplace_back(worker, t);
  for (auto& t : ts) t.join();
}

// ----------------------------------------------------------------------------
// src/prune.rs:64-120  run_e_step.  Snippets of MAX_SAMPLE_LENGTH = 8192*10
// bytes (:75,83); z must be "normal" (:90-96).  Partial sums are merged in
// CHUNK INDEX order here (the reference merges in rayon completion order — the
// one place it is itself non-deterministic, at the 1e-16 level).
// literal != 0 → build the Lattice and call populate_marginal exactly as the
// reference does; literal == 0 → per-position form (bit-identical, faster).
// ----------------------------------------------------------------------------
static int run_e_step(const Model& m, const uint8_t* blob, const uint64_t* off, size_t S,
                      int threads, int literal, size_t max_sample_length, double* expected_out,
                      int64_t* bad_sample, double* bad_z, double dropout = 0.0, const KeyedDraw* keyed = nullptr,
                      uint64_t byte_base = 0, uint64_t* fixed_out = nullptr) {
  size_t V = m.vocab_size();
  size_t chunk = par_chunk_size(S, (size_t)std::max(1, threads), 8);  // :66
  size_t n_chunks = S ? (S + chunk - 1) / chunk : 0;
  std::vector<std::vector<double>> partial(n_chunks);
  std::vector<std::vector<uint64_t>> partial_fixed(fixed_out ? n_chunks : 0);  // exact sums (fixed_out != null)
  std::atomic<int64_t> bad{-1};
  std::mutex bad_mu;
  double badz = 0.0;
  parallel_chunks(S, chunk, threads, [&](size_t c, size_t lo, size_t hi, int) {
    std::vector<double>& ef = partial[c];
    ef.assign(V, 0.0);  // :78
    MarginalSinks sinks;
    if (fixed_out) {
      partial_fixed[c].assign(3 * V, 0);
      sinks.fixed = partial_fixed[c].data();
    }
    const MarginalSinks* sk = fixed_out ? &sinks : nullptr;
    Lattice lat;
    std::vector<double> A, B;
    std::vector<uint8_t> seen;
    uint64_t rng = 0;
    for (size_t s = lo; s < hi; s++) {
      const uint8_t* p = blob + off[s];
      size_t n = off[s + 1] - off[s];
      for (size_t o = 0; o < n; o += max_sample_length) {  // :83 sample.as_bytes().chunks(MAX)
        size_t sn = std::min(max_sample_length, n - o);
        double z;
        if (literal || dropout > 0.0) {
          lat.from(p + o, sn);
          populate_nodes(m, lat, dropout, &rng, keyed, byte_base + off[s] + o);  // :87
          z = populate_marginal(lat, ef.data(), sk);
        } else {
          z = marginal_per_position(m, p + o, sn, ef.data(), A, B, seen, sk);
        }
        if (!std::isnormal(z)) {  // :90-96 panic
          std::lock_guard<std::mutex> g(bad_mu);
          if (bad.load() < 0 || (int64_t)s < bad.load()) { bad.store((int64_t)s); badz = z; }
        }
      }
    }
  });
  for (size_t i = 0; i < V; i++) expected_out[i] = 0.0;
  for (size_t c = 0; c < n_chunks; c++)  // :104-112
    for (size_t i = 0; i < V; i++) expected_out[i] += partial[c][i];
  if (fixed_out) {  // integer additions: the merge order does not matter
    std::fill(fixed_out, fixed_out + 3 * V, 0);
    for (size_t c = 0; c < n_chunks; c++)
      for (size_t i = 0; i < V; i++) fixed_merge(fixed_out + 3 * i, partial_fixed[c].data() + 3 * i);
  }
  *bad_sample = bad.load();
  *bad_z = badz;
  return bad.load() >= 0 ? 1 : 0;
}

// src/prune.rs:322-335  digamma
static double digamma(double x) {
  double result = 0.0;
  while (x < 7.0) {
    result -= 1.0 / x;
    x += 1.0;
  }
  x -= 1.0 / 2.0;
  double xx = 1.0 / x;
  double xx2 = xx * xx;
  double xx4 = xx2 * xx2;
  result += std::log(x) + (1.0 / 24.0) * xx2 - 7.0 / 960.0 * xx4 + (31.0 / 8064.0) * xx4 * xx2 -
            (127.0 / 30720.0) * xx4 * xx4;
  return result;
}

// src/prune.rs:124-170  run_m_step.  Returns 1 if a score is NaN/inf (panic).
static int run_m_step(const Model& m, const double* expected, std::vector<ScoredToken>& out) {
  const double THRESH = 0.5;  // :127
  out.clear();
  for (size_t i = 0; i < m.vocab_size(); i++) {  // :131-138
    double freq = expected[i];
    const ScoredToken& t = m.vocab[i];
    if (freq < THRESH && !t.keep) continue;
    out.push_back(ScoredToken{t.value, std::fmax(freq, THRESH), t.keep});
  }
  double sum = 0.0;  // :143-146  iter().map().sum::<f64>()  (sequential left fold from 0.0)
  for (auto& t : out) sum += t.score;
  double logsum = digamma(sum);  // :147
  int bad = 0;
  for (auto& t : out) {
    double s = digamma(t.score) - logsum;  // :148-151
    if (std::isnan(s) || std::isinf(s)) bad = 1;  // :154-163
    t.score = s;
  }
  return bad;
}

// ----------------------------------------------------------------------------
// src/prune.rs:173-319  prune_vocab.
// sort_unstable_by has reference-undefined order among exact ties; here ties
// are broken deterministically (candidates: id ascending; final vocab: prior
// index ascending) and `n_loss_ties_at_cut` reports whether a tie straddled the
// cut, so a set mismatch can be attributed (SURVEY.md H6).
// Return: 0 ok, 1 NoPath in the frequency pass, 2 non-normal loss (panic :291).
// ----------------------------------------------------------------------------
struct PruneAudit {
  uint64_t n_always_keep_false = 0, n_with_alternatives = 0, n_silent_drop = 0, n_zero_freq_drop = 0,
           n_candidates = 0, n_loss_ties_at_cut = 0;
  double min_loss_gap_at_cut = 0.0;
};

static void token_alternatives(const Model& m, std::vector<uint8_t>& always_keep,
                               std::vector<std::vector<uint32_t>>& alternatives) {
  size_t V = m.vocab_size();
  always_keep.assign(V, 1);
  alternatives.assign(V, {});
  Lattice lat;
  uint64_t rng = 0;
  for (size_t id = 0; id < V; id++) {  // :183-203
    const auto& tok = m.vocab[id];
    lat.from(tok.value.data(), tok.value.size());
    populate_nodes(m, lat, 0.0, &rng);
    auto nbests = nbest(lat, 2);
    if (nbests.size() > 1 && nbests[0].size() > 1) always_keep[id] = 0;  // :191-195
    if (nbests.size() > 1 && nbests[0].size() == 1) {                    // :197-202
      for (size_t ni : nbests[1]) alternatives[id].push_back(lat.nodes[ni].token_id);
    }
  }
}

static int token_frequencies(const Model& m, const uint8_t* blob, const uint64_t* off, size_t S,
                             int threads, std::vector<uint64_t>& freq, uint64_t* err_pos,
                             uint64_t* err_len) {
  size_t V = m.vocab_size();
  size_t chunk = par_chunk_size(S, (size_t)std::max(1, threads), 2);  // :206
  size_t n_chunks = S ? (S + chunk - 1) / chunk : 0;
  std::vector<std::vector<uint64_t>> partial(n_chunks);
  std::atomic<int> err{0};
  std::mutex mu;
  parallel_chunks(S, chunk, threads, [&](size_t c, size_t lo, size_t hi, int) {
    auto& f = partial[c];
    f.assign(V, 0);
    std::vector<uint32_t> ids;
    uint64_t rng = 0;
    for (size_t s = lo; s < hi; s++) {
      uint64_t ep = 0, el = 0;
      int rc = encode(m, blob + off[s], off[s + 1] - off[s], 0.0, ids, &ep, &el, &rng);  // :218
      if (rc) {
        std::lock_guard<std::mutex> g(mu);
        if (!err.load()) { err.store(1); *err_pos = ep; *err_len = el; }
        return;
      }
      for (uint32_t id : ids) f[id] += 1;  // :223-225
    }
  });
  freq.assign(V, 0);
  for (size_t c = 0; c < n_chunks; c++)
    for (size_t i = 0; i < V; i++) freq[i] += partial[c][i];
  return err.load();
}

// ----------------------------------------------------------------------------
// src/merge.rs:36-84  pair-frequency pass of ModelVocabularyMerger::merge:
// encode every sample (dropout 0.0) and count adjacent id pairs within the sample
// (chunk-local FnvHashMaps merged under a lock), then `pairs.sort_unstable_by(|a, b|
// b.1.cmp(&a.1))`.  sort_unstable leaves the order of equal frequencies undefined;
// here ties are ordered by (first id, second id) ascending.
// ----------------------------------------------------------------------------
static int pair_frequencies(const Model& m, const uint8_t* blob, const uint64_t* off, size_t S, int threads,
                            std::vector<std::pair<uint64_t, uint64_t>>& out, uint64_t* err_pos, uint64_t* err_len) {
  size_t chunk = par_chunk_size(S, (size_t)std::max(1, threads), 4);  // :41
  std::unordered_map<uint64_t, uint64_t> all;
  std::atomic<int> err{0};
  std::mutex mu;
  parallel_chunks(S, chunk, threads, [&](size_t, size_t lo, size_t hi, int) {
    std::unordered_map<uint64_t, uint64_t> local;  // :56
    std::vector<uint32_t> ids;
    uint64_t rng = 0;
    for (size_t s = lo; s < hi; s++) {
      uint64_t ep = 0, el = 0;
      int rc = encode(m, blob + off[s], off[s + 1] - off[s], 0.0, ids, &ep, &el, &rng);  // :59 (.unwrap())
      if (rc) {
        std::lock_guard<std::mutex> g(mu);
        if (!err.load()) { err.store(1); *err_pos = ep; *err_len = el; }
        return;
      }
      for (size_t i = 1; i < ids.size(); i++)  // :61-64
        local[((uint64_t)ids[i - 1] << 32) | ids[i]] += 1;
    }
    std::lock_guard<std::mutex> g(mu);  // :69-74
    for (auto& kv : local) all[kv.first] += kv.second;
  });
  out.assign(all.begin(), all.end());
  std::sort(out.begin(), out.end(), [](const std::pair<uint64_t, uint64_t>& a, const std::pair<uint64_t, uint64_t>& b) {
    if (a.second != b.second) return a.second > b.second;  // :83
    return a.first < b.first;
  });
  return err.load();
}

static int prune_vocab(const Model& m, const uint8_t* blob, const uint64_t* off, size_t S,
                       int threads, size_t target_vocab_size, double shrink_factor,
                       std::vector<ScoredToken>& pruned_vocab, PruneAudit* audit) {
  size_t V = m.vocab_size();
  size_t pruned_size = (size_t)((double)V * shrink_factor);  // :174
  pruned_size = std::max(pruned_size, target_vocab_size);    // :175
  std::vector<uint8_t> always_keep;
  std::vector<std::vector<uint32_t>> alternatives;
  token_alternatives(m, always_keep, alternatives);
  std::vector<uint64_t> token_frequencies_v;
  uint64_t ep = 0, el = 0;
  if (token_frequencies(m, blob, off, S, threads, token_frequencies_v, &ep, &el)) return 1;

  uint64_t sum_u = 0;
  for (uint64_t f : token_frequencies_v) sum_u += f;
  double sum_token_frequencies = (double)sum_u;                    // :248
  double logsum_token_frequencies = std::log(sum_token_frequencies);  // :249

  std::vector<std::pair<size_t, double>> candidates;
  pruned_vocab.clear();
  PruneAudit au;
  for (size_t id = 0; id < V; id++) {  // :260-300
    const ScoredToken& token = m.vocab[id];
    if (!always_keep[id]) au.n_always_keep_false++;
    if (!alternatives[id].empty()) au.n_with_alternatives++;
    if (token.keep) { pruned_vocab.push_back(token); continue; }
    if (token_frequencies_v[id] == 0 && !always_keep[id]) {
      au.n_zero_freq_drop++;
      continue;
    } else if (alternatives[id].empty()) {
      pruned_vocab.push_back(token);
    } else if (token_frequencies_v[id] != 0) {
      double freq = (double)token_frequencies_v[id];
      double logprob = std::log(freq) - logsum_token_frequencies;
      // :279  alternatives.len() is the OUTER vector's length = V  (quirk Q14)
      double alt_logsum = std::log(sum_token_frequencies + freq * (double)(alternatives.size() - 1));
      double alt_logprob = 0.0;
      for (uint32_t alt_id : alternatives[id])
        alt_logprob += std::log((double)token_frequencies_v[alt_id] + freq) - alt_logsum;
      double loss = (freq / (double)S) * (logprob - alt_logprob);  // :290
      if (!std::isnormal(loss)) return 2;                          // :291-296
      candidates.emplace_back(id, loss);
    } else {
      au.n_silent_drop++;  // freq==0 && always_keep && has alternatives: falls through (Q14)
    }
  }
  au.n_candidates = candidates.size();
  // :308  sort_unstable_by(|(_,a),(_,b)| b.partial_cmp(a))  → loss descending
  std::stable_sort(candidates.begin(), candidates.end(),
                   [](const auto& a, const auto& b) { return a.second > b.second; });
  size_t taken = 0;
  for (auto& c : candidates) {  // :309-314
    if (pruned_vocab.size() == pruned_size) break;
    pruned_vocab.push_back(m.vocab[c.first]);
    taken++;
  }
  if (taken > 0 && taken < candidates.size()) {
    double a = candidates[taken - 1].second, b = candidates[taken].second;
    au.min_loss_gap_at_cut = a - b;
    if (a == b) au.n_loss_ties_at_cut = 1;
  }
  // :316  sort_unstable_by(|a,b| b.score.partial_cmp(&a.score))  → score descending
  std::stable_sort(pruned_vocab.begin(), pruned_vocab.end(),
                   [](const ScoredToken& a, const ScoredToken& b) { return a.score > b.score; });
  if (audit) *audit = au;
  return 0;
}

}  // namespace orc

// =============================================================================
// C interface for ctypes (tests / bench only)
// =============================================================================
using namespace orc;

struct orc_model {
  std::unique_ptr<Model> m;
};

static std::vector<ScoredToken> make_vocab(const uint8_t* bytes, const uint64_t* off,
                                           const double* scores, const uint8_t* keep, uint64_t V) {
  std::vector<ScoredToken> v;
  v.reserve(V);
  for (uint64_t i = 0; i < V; i++)
    v.push_back(ScoredToken{std::vector<uint8_t>(bytes + off[i], bytes + off[i + 1]), scores[i],
                            keep ? keep[i] != 0 : false});
  return v;
}

static void export_vocab(const std::vector<ScoredToken>& v, uint8_t* bytes, uint64_t* off,
                         double* scores, uint8_t* keep) {
  uint64_t o = 0;
  for (size_t i = 0; i < v.size(); i++) {
    off[i] = o;
    if (!v[i].value.empty()) std::memcpy(bytes + o, v[i].value.data(), v[i].value.size());
    o += v[i].value.size();
    scores[i] = v[i].score;
    keep[i] = v[i].keep;
  }
  off[v.size()] = o;
}

extern "C" {

orc_model* orc_model_create(const uint8_t* bytes, const uint64_t* off, const double* scores,
                            const uint8_t* keep, uint64_t V) {
  auto* h = new orc_model();
  h->m.reset(new Model(make_vocab(bytes, off, scores, keep, V)));
  return h;
}
void orc_model_destroy(orc_model* h) { delete h; }
uint64_t orc_model_vocab_size(orc_model* h) { return h->m->vocab_size(); }
uint64_t orc_model_vocab_bytes(orc_model* h) {
  uint64_t n = 0;
  for (auto& t : h->m->vocab) n += t.value.size();
  return n;
}
void orc_model_export(orc_model* h, uint8_t* bytes, uint64_t* off, double* scores, uint8_t* keep) {
  export_vocab(h->m->vocab, bytes, off, scores, keep);
}

// Model::encode.  Returns #ids, or -1 for NoPath (err[0]=pos, err[1]=len).
int64_t orc_encode(orc_model* h, const uint8_t* text, uint64_t n, double dropout, uint32_t* out,
                   uint64_t cap, uint64_t* err) {
  std::vector<uint32_t> ids;
  uint64_t ep = 0, el = 0;
  int rc = encode(*h->m, text, n, dropout, ids, &ep, &el, &h->m->rng_state);
  if (rc) { err[0] = ep; err[1] = el; return -1; }
  if (ids.size() > cap) return -2;
  std::memcpy(out, ids.data(), ids.size() * 4);
  return (int64_t)ids.size();
}

// Model::encode with the keyed dropout draw of tgx_model_set_dropout (sample = index of this text in the call).
int64_t orc_encode_keyed(orc_model* h, const uint8_t* text, uint64_t n, double dropout, uint64_t seed,
                         uint64_t sample, uint32_t* out, uint64_t cap, uint64_t* err) {
  std::vector<uint32_t> ids;
  uint64_t ep = 0, el = 0;
  KeyedDraw kd(seed, sample);
  int rc = encode(*h->m, text, n, dropout, ids, &ep, &el, &h->m->rng_state, &kd);
  if (rc) { err[0] = ep; err[1] = el; return -1; }
  if (ids.size() > cap) return -2;
  std::memcpy(out, ids.data(), ids.size() * 4);
  return (int64_t)ids.size();
}

uint64_t orc_crlf(const uint8_t* s, uint64_t n, uint8_t* out) { return crlf(s, n, out); }

// Tokenizer::encode_ordinary_batch (src/tokenizer.rs:114-123) with an optional
// crlf processor: per-sample (rayon into_par_iter → dynamic per-sample
// scheduling over `threads` workers), outputs in input order.  id_off[S+1].
// status[s] = 0 ok / 1 NoPath; proc_len[s] = processed length.  Returns the
// lowest failing sample index + 1, or 0.
uint64_t orc_encode_batch(orc_model* h, const uint8_t* blob, const uint64_t* off, uint64_t S,
                          int use_crlf, int threads, uint32_t* ids_out, uint64_t cap,
                          uint64_t* id_off, int32_t* status, uint64_t* proc_len) {
  std::vector<std::vector<uint32_t>> res(S);
  std::vector<int32_t> st(S, 0);
  std::vector<uint64_t> pl(S, 0);
  parallel_chunks(S, 1, threads, [&](size_t, size_t lo, size_t hi, int) {
    std::vector<uint8_t> buf;
    uint64_t rng = 0;
    for (size_t s = lo; s < hi; s++) {
      const uint8_t* p = blob + off[s];
      size_t n = off[s + 1] - off[s];
      if (use_crlf) {  // processors.fold(input.to_string(), |s,p| p.preprocess(&s))  :115-118
        buf.resize(n ? n : 1);
        n = crlf(p, n, buf.data());
        p = buf.data();
      }
      uint64_t ep, el;
      st[s] = encode(*h->m, p, n, 0.0, res[s], &ep, &el, &rng);
      pl[s] = n;
    }
  });
  uint64_t o = 0, first_bad = 0;
  for (uint64_t s = 0; s < S; s++) {
    id_off[s] = o;
    if (status) status[s] = st[s];
    if (proc_len) proc_len[s] = pl[s];
    if (st[s] && !first_bad) first_bad = s + 1;
    if (o + res[s].size() <= cap && !res[s].empty())
      std::memcpy(ids_out + o, res[s].data(), res[s].size() * 4);
    o += res[s].size();
  }
  id_off[S] = o;
  return first_bad;
}

// Trie common_prefix_search (src/model.rs:132-138): ids of all tokens prefixing text.
uint64_t orc_common_prefix_search(orc_model* h, const uint8_t* text, uint64_t n, uint32_t* ids,
                                  uint32_t* lens, uint64_t cap) {
  uint64_t k = 0;
  common_prefix_search(h->m->trie, text, n, [&](uint32_t id, uint32_t len) {
    if (k < cap) { ids[k] = id; lens[k] = len; }
    k++;
  });
  return k;
}

// One lattice: populate_nodes + populate_marginal on a single sentence.
// expected[V] is accumulated into (+=).  literal: see run_e_step.
double orc_marginal(orc_model* h, const uint8_t* s, uint64_t n, double* expected, int literal) {
  if (literal) {
    Lattice lat;
    uint64_t rng = 0;
    lat.from(s, n);
    populate_nodes(*h->m, lat, 0.0, &rng);
    return populate_marginal(lat, expected);
  }
  std::vector<double> A, B;
  std::vector<uint8_t> seen;
  return marginal_per_position(*h->m, s, n, expected, A, B, seen);
}

// A[0..n] and B[0..n] of the per-position form (debug aid for kernel tests).
double orc_alpha_beta(orc_model* h, const uint8_t* s, uint64_t n, double* A_out, double* B_out) {
  std::vector<double> A, B, ex(h->m->vocab_size(), 0.0);
  std::vector<uint8_t> seen;
  double z = marginal_per_position(*h->m, s, n, ex.data(), A, B, seen);
  std::memcpy(A_out, A.data(), (n + 1) * 8);
  std::memcpy(B_out, B.data(), (n + 1) * 8);
  return z;
}

int orc_run_e_step(orc_model* h, const uint8_t* blob, const uint64_t* off, uint64_t S, int threads,
                   int literal, uint64_t max_sample_length, double* expected, int64_t* bad_sample,
                   double* bad_z) {
  return run_e_step(*h->m, blob, off, S, threads, literal, max_sample_length, expected, bad_sample,
                    bad_z);
}

// run_e_step with populate_nodes(.., dropout) (src/prune.rs:87).  keyed != 0: the product's keyed draw (key = seed,
// position = byte_base + byte offset in `blob`); keyed == 0: a sequential splitmix64 per rayon chunk, i.e. the
// reference's loop with a seeded generator.
int orc_run_e_step_dropout(orc_model* h, const uint8_t* blob, const uint64_t* off, uint64_t S, int threads,
                           uint64_t max_sample_length, double dropout, int keyed, uint64_t seed, uint64_t byte_base,
                           double* expected, int64_t* bad_sample, double* bad_z) {
  KeyedDraw kd(seed, ~0ull);
  return run_e_step(*h->m, blob, off, S, threads, 1, max_sample_length, expected, bad_sample, bad_z, dropout,
                    keyed ? &kd : nullptr, byte_base);
}

// run_e_step (dropout 0: the plain E-step; else as orc_run_e_step_dropout) with the exact sums beside the f64 ones:
// fixed[3 * id + 0 / 1 / 2] = bits 65..128 / bits 1..64 / integer part of sum(floor(c * 2^128)) over token id's
// contributions c.  The integer sums do not depend on the thread count or the order of the additions.
int orc_run_e_step_fixed(orc_model* h, const uint8_t* blob, const uint64_t* off, uint64_t S, int threads,
                         uint64_t max_sample_length, double dropout, int keyed, uint64_t seed, uint64_t byte_base,
                         uint64_t* fixed, int64_t* bad_sample, double* bad_z) {
  KeyedDraw kd(seed, ~0ull);
  std::vector<double> ex(h->m->vocab_size());
  return run_e_step(*h->m, blob, off, S, threads, dropout > 0.0 ? 1 : 0, max_sample_length, ex.data(), bad_sample,
                    bad_z, dropout, keyed ? &kd : nullptr, byte_base, fixed);
}

// The contributions (id, exp(a + score + b - z)) of one lattice (populate_nodes + populate_marginal) in the order the
// reference adds them.  dropout > 0: the keyed draw of orc_run_e_step_fixed, with the lattice's first byte at position
// byte_base.  Writes at most cap of them; *count = their number.  Returns z.
double orc_marginal_contributions(orc_model* h, const uint8_t* s, uint64_t n, uint32_t* ids_out, double* vals_out,
                                  uint64_t cap, uint64_t* count, double dropout, uint64_t seed, uint64_t byte_base) {
  Lattice lat;
  uint64_t rng = 0;
  KeyedDraw kd(seed, ~0ull);
  lat.from(s, n);
  populate_nodes(*h->m, lat, dropout, &rng, &kd, byte_base);
  std::vector<double> ex(h->m->vocab_size(), 0.0);
  std::vector<std::pair<uint32_t, double>> cs;
  MarginalSinks sinks;
  sinks.contribs = &cs;
  const double z = populate_marginal(lat, ex.data(), &sinks);
  for (size_t i = 0; i < cs.size() && i < cap; i++) {
    ids_out[i] = cs[i].first;
    vals_out[i] = cs[i].second;
  }
  *count = cs.size();
  return z;
}

double orc_digamma(double x) { return digamma(x); }
double orc_log_sum_exp(double x, double y, int init) { return log_sum_exp(x, y, init != 0); }

// run_m_step → new model handle (Model::from(vocab), src/prune.rs:48).  rc in *rc.
orc_model* orc_run_m_step(orc_model* h, const double* expected, int* rc) {
  std::vector<ScoredToken> out;
  *rc = run_m_step(*h->m, expected, out);
  auto* nh = new orc_model();
  nh->m.reset(new Model(std::move(out)));
  return nh;
}

int orc_token_frequencies(orc_model* h, const uint8_t* blob, const uint64_t* off, uint64_t S,
                          int threads, uint64_t* freq, uint64_t* err) {
  std::vector<uint64_t> f;
  int rc = token_frequencies(*h->m, blob, off, S, threads, f, &err[0], &err[1]);
  if (!rc) std::memcpy(freq, f.data(), f.size() * 8);
  return rc;
}

// pairs[i] = (first id << 32) | second id, counts[i]; frequency-descending.  Returns the number of distinct
// pairs (writes at most cap of them), or -1 on NoPath (err = pos, len).
int64_t orc_pair_frequencies(orc_model* h, const uint8_t* blob, const uint64_t* off, uint64_t S, int threads,
                             uint64_t* pairs, uint64_t* counts, uint64_t cap, uint64_t* err) {
  std::vector<std::pair<uint64_t, uint64_t>> v;
  if (pair_frequencies(*h->m, blob, off, S, threads, v, &err[0], &err[1])) return -1;
  for (size_t i = 0; i < v.size() && i < cap; i++) {
    pairs[i] = v[i].first;
    counts[i] = v[i].second;
  }
  return (int64_t)v.size();
}

// always_keep[V] and alternatives (CSR: alt_off[V+1], alt_ids[cap]) of prune_vocab.
uint64_t orc_token_alternatives(orc_model* h, uint8_t* always_keep, uint64_t* alt_off,
                                uint32_t* alt_ids, uint64_t cap) {
  std::vector<uint8_t> ak;
  std::vector<std::vector<uint32_t>> alts;
  token_alternatives(*h->m, ak, alts);
  uint64_t o = 0;
  for (size_t i = 0; i < ak.size(); i++) {
    always_keep[i] = ak[i];
    alt_off[i] = o;
    for (uint32_t a : alts[i]) {
      if (o < cap) alt_ids[o] = a;
      o++;
    }
  }
  alt_off[ak.size()] = o;
  return o;
}

// nbest on one sentence: returns number of paths; path k = ids[path_off[k]..path_off[k+1]).
uint64_t orc_nbest(orc_model* h, const uint8_t* s, uint64_t n, uint64_t nb, uint32_t* ids,
                   uint64_t* path_off, uint64_t cap) {
  Lattice lat;
  uint64_t rng = 0;
  lat.from(s, n);
  populate_nodes(*h->m, lat, 0.0, &rng);
  auto paths = nbest(lat, nb);
  uint64_t o = 0;
  for (size_t k = 0; k < paths.size(); k++) {
    path_off[k] = o;
    for (size_t ni : paths[k]) {
      if (o < cap) ids[o] = lat.nodes[ni].token_id;
      o++;
    }
  }
  path_off[paths.size()] = o;
  return paths.size();
}

// prune_vocab → new model handle.  audit[8]: see PruneAudit.
orc_model* orc_prune_vocab(orc_model* h, const uint8_t* blob, const uint64_t* off, uint64_t S,
                           int threads, uint64_t target, double shrink, int* rc, double* audit) {
  std::vector<ScoredToken> out;
  PruneAudit au;
  *rc = prune_vocab(*h->m, blob, off, S, threads, target, shrink, out, &au);
  if (audit) {
    audit[0] = (double)au.n_always_keep_false;
    audit[1] = (double)au.n_with_alternatives;
    audit[2] = (double)au.n_silent_drop;
    audit[3] = (double)au.n_zero_freq_drop;
    audit[4] = (double)au.n_candidates;
    audit[5] = (double)au.n_loss_ties_at_cut;
    audit[6] = au.min_loss_gap_at_cut;
  }
  auto* nh = new orc_model();
  nh->m.reset(new Model(std::move(out)));
  return nh;
}

// src/prune.rs:23-57  ModelVocabularyPruner::prune — full loop.  Returns the
// final model; *rc != 0 on panic/NoPath; iters[] receives vocab sizes after
// every E/M sub-iteration and prune step (up to cap entries), *n_iters count.
orc_model* orc_prune(orc_model* h, const uint8_t* blob, const uint64_t* off, uint64_t S, int threads,
                     uint64_t vocab_size, double shrink, uint64_t em_subiters, int* rc,
                     uint64_t* iters, uint64_t cap, uint64_t* n_iters) {
  std::unique_ptr<Model> model(new Model(h->m->vocab));
  *rc = 0;
  uint64_t k = 0;
  while (model->vocab_size() > vocab_size) {
    for (uint64_t sub = 0; sub < em_subiters; sub++) {
      std::vector<double> expected(model->vocab_size());
      int64_t bad;
      double badz;
      if (run_e_step(*model, blob, off, S, threads, 0, 8192 * 10, expected.data(), &bad, &badz)) {
        *rc = 3;
        goto done;
      }
      std::vector<ScoredToken> v;
      if (run_m_step(*model, expected.data(), v)) { *rc = 4; goto done; }
      model.reset(new Model(std::move(v)));
      if (k < cap) iters[k] = model->vocab_size();
      k++;
    }
    {
      std::vector<ScoredToken> v;
      int prc = prune_vocab(*model, blob, off, S, threads, vocab_size, shrink, v, nullptr);
      if (prc) { *rc = prc; goto done; }
      model.reset(new Model(std::move(v)));
      if (k < cap) iters[k] = model->vocab_size();
      k++;
    }
  }
done:
  *n_iters = k;
  auto* nh = new orc_model();
  nh->m = std::move(model);
  return nh;
}

}  // extern "C"
