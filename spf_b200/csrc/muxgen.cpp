// muxgen.cpp -- host-side generator of the MUX circuits Parasol instructions expand into
// (SURVEY.md 8(f).3: the step before the hot path).  The reference builds one reduced ordered BDD
// per output bit with biodivine-lib-bdd, turns every BDD node into a multiplexer
// (mux_circuits/src/lib.rs:355-451, From<&[Bdd]>), and for the big circuits merges duplicates by
// common-subexpression elimination (lib.rs:249-252); it ships the 8x8/16x16 multipliers and the
// 64x64 reduction as pre-generated blobs because that takes long (mul.rs:62-68,393-400).
//
// Here ONE shared ROBDD manager (unique table + computed cache) holds all output functions of a
// circuit, so sub-functions are shared between outputs from the start, and the (duplicated-variable
// -> real input) renaming of the multiplier is a single bottom-up re-hash.  The functions follow the
// reference's constructions line by line in meaning (cited per function) so that the circuits
// compute the same Boolean functions over the same input order; node numbering differs, and this
// generator never emits a multiplexer whose two data inputs coincide.
//
// Pure host code, no CUDA: callable on a box without a GPU.
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <unordered_map>
#include <vector>

#include "../../include/spf_b200.h"

namespace {

struct BddManager {
  struct Node { uint32_t var, lo, hi; };
  std::vector<Node> nodes;           // 0 = false, 1 = true; children precede parents
  std::vector<uint32_t> table;       // open-addressing unique table of node ids (0 = empty)
  size_t table_mask = 0, table_used = 0;
  struct CacheEntry { uint32_t a, b, op, r; };
  std::vector<CacheEntry> cache;     // direct-mapped, lossy computed cache
  uint32_t nvars;
  bool overflow = false;
  enum { AND = 1, OR = 2, XOR = 3 };
  static constexpr uint32_t kMaxNodes = 1u << 28;

  explicit BddManager(uint32_t nv) : nvars(nv) {
    nodes.push_back({nv, 0, 0});
    nodes.push_back({nv, 1, 1});
    table.assign(1u << 16, 0);
    table_mask = table.size() - 1;
    cache.assign(1u << 20, CacheEntry{0, 0, 0, 0});
  }
  static uint64_t mix(uint64_t a, uint64_t b, uint64_t c) {
    uint64_t h = a * 0x9E3779B97F4A7C15ull ^ (b + 0x7F4A7C15ull) * 0xC2B2AE3D27D4EB4Full ^ (c + 0x165667B1ull) * 0xD6E8FEB86659FD93ull;
    h ^= h >> 29; h *= 0xBF58476D1CE4E5B9ull; h ^= h >> 32;
    return h;
  }
  void grow() {
    std::vector<uint32_t> t(table.size() * 2, 0);
    const size_t mask = t.size() - 1;
    for (uint32_t id : table) {
      if (!id) continue;
      size_t h = mix(nodes[id].var, nodes[id].lo, nodes[id].hi) & mask;
      while (t[h]) h = (h + 1) & mask;
      t[h] = id;
    }
    table.swap(t);
    table_mask = mask;
  }
  uint32_t mk(uint32_t var, uint32_t lo, uint32_t hi) {
    if (lo == hi) return lo;
    size_t h = mix(var, lo, hi) & table_mask;
    while (uint32_t id = table[h]) {
      const Node& n = nodes[id];
      if (n.var == var && n.lo == lo && n.hi == hi) return id;
      h = (h + 1) & table_mask;
    }
    if (nodes.size() >= kMaxNodes) { overflow = true; return 0; }
    const uint32_t id = (uint32_t)nodes.size();
    nodes.push_back({var, lo, hi});
    table[h] = id;
    if (++table_used * 2 > table.size()) grow();
    return id;
  }
  uint32_t var(uint32_t v) { return mk(v, 0, 1); }
  uint32_t apply(uint32_t op, uint32_t a, uint32_t b) {
    if (a > b) std::swap(a, b);  // all three operators commute
    switch (op) {
      case AND: if (a == 0) return 0; if (a == 1) return b; if (a == b) return a; break;
      case OR: if (a == 1) return 1; if (a == 0) return b; if (a == b) return a; break;
      default: if (a == 0) return b; if (a == b) return 0; break;  // XOR; a == 1 is negation, recursed
    }
    CacheEntry& e = cache[mix(a, b, op) & (cache.size() - 1)];
    if (e.op == op && e.a == a && e.b == b) return e.r;
    const Node na = nodes[a], nb = nodes[b];
    const uint32_t v = std::min(na.var, nb.var);
    const uint32_t a0 = na.var == v ? na.lo : a, a1 = na.var == v ? na.hi : a;
    const uint32_t b0 = nb.var == v ? nb.lo : b, b1 = nb.var == v ? nb.hi : b;
    const uint32_t r0 = apply(op, a0, b0);
    const uint32_t r1 = apply(op, a1, b1);
    const uint32_t r = mk(v, r0, r1);
    CacheEntry& e2 = cache[mix(a, b, op) & (cache.size() - 1)];
    e2 = {a, b, op, r};
    return r;
  }
  uint32_t band(uint32_t a, uint32_t b) { return apply(AND, a, b); }
  uint32_t bor(uint32_t a, uint32_t b) { return apply(OR, a, b); }
  uint32_t bxor(uint32_t a, uint32_t b) { return apply(XOR, a, b); }
  uint32_t bnot(uint32_t a) { return apply(XOR, a, 1); }
  uint32_t and_not(uint32_t a, uint32_t b) { return band(a, bnot(b)); }
};

typedef std::vector<uint32_t> Fns;

// ---- the reference's constructions ---------------------------------------------------------------

// ripple_carry_adder (mux_circuits/src/add.rs:13-56): inputs [cin] a0 b0 a1 b1 ... then the rest of
// the longer operand; outputs max(n, m) sum bits then the carry.
Fns build_adder(BddManager& M, uint32_t n, uint32_t m, bool cin) {
  const uint32_t lo = std::min(n, m), hi = std::max(n, m), off = cin ? 1 : 0;
  uint32_t carry = cin ? M.var(0) : 0;
  Fns sum(hi + 1, 1);
  for (uint32_t i = 0; i < lo; i++) {
    const uint32_t a = M.var(off + 2 * i), b = M.var(off + 2 * i + 1), axb = M.bxor(a, b);
    sum[i] = M.bxor(carry, axb);
    carry = M.bor(M.band(axb, carry), M.band(a, b));
  }
  for (uint32_t i = 0; i < hi - lo; i++) {
    const uint32_t a = M.var(2 * lo + i + off);
    sum[i + lo] = M.bxor(carry, a);
    carry = M.band(a, carry);
  }
  sum[hi] = carry;
  return sum;
}

// full_subtractor (sub.rs:12-49): inputs [bin] a0 b0 a1 b1 ...; outputs n difference bits then the borrow.
Fns build_subtractor(BddManager& M, uint32_t n, bool bin) {
  const uint32_t off = bin ? 1 : 0;
  uint32_t borrow = bin ? M.var(0) : 0;
  Fns diff(n + 1, 1);
  for (uint32_t i = 0; i < n; i++) {
    const uint32_t a = M.var(off + 2 * i), b = M.var(off + 2 * i + 1), axb = M.bxor(a, b);
    diff[i] = M.bxor(borrow, axb);
    borrow = M.bor(M.and_not(borrow, axb), M.and_not(b, a));
  }
  diff[n] = borrow;
  return diff;
}

// negator (neg.rs:7-27): two's complement, copy bits up to and including the first 1, flip the rest.
Fns build_negator(BddManager& M, uint32_t n) {
  uint32_t flip = 0;
  Fns neg(n, 1);
  for (uint32_t i = 0; i < n; i++) {
    neg[i] = M.bxor(flip, M.var(i));
    flip = M.bor(flip, M.var(i));
  }
  return neg;
}

// unsigned_comparison_impl (comparisons.rs:143-181) over interleaved inputs a0 b0 a1 b1 ...
uint32_t unsigned_compare(BddManager& M, uint32_t pairs, bool greater, bool or_equal) {
  uint32_t result = 0, all_equal = 1;
  for (uint32_t i = pairs; i-- > 0;) {
    const uint32_t a = M.var(2 * i), b = M.var(2 * i + 1);
    const uint32_t cmp = greater ? M.and_not(a, b) : M.and_not(b, a);
    result = M.bor(result, M.band(cmp, all_equal));
    all_equal = M.band(all_equal, M.bnot(M.bxor(a, b)));
  }
  if (or_equal) result = M.bor(result, all_equal);
  return result;
}

// compare_or_maybe_equal_signed (comparisons.rs:79-117): the sign bits override the unsigned result
// of the lower n - 1 bit pairs.
uint32_t signed_compare(BddManager& M, uint32_t n, bool greater, bool or_equal) {
  const uint32_t a = M.var(2 * n - 2), b = M.var(2 * n - 1);
  const uint32_t a_lt_b = M.and_not(b, a), a_gt_b = M.and_not(a, b);
  const uint32_t force_true = greater ? a_lt_b : a_gt_b, force_false = greater ? a_gt_b : a_lt_b;
  const uint32_t r = unsigned_compare(M, n - 1, greater, or_equal);
  return M.and_not(M.bor(r, force_true), force_false);
}

// compare_equal / compare_not_equal (comparisons.rs:19-72)
uint32_t all_pairs_equal(BddManager& M, uint32_t n) {
  uint32_t r = 1;
  for (uint32_t i = 0; i < n; i++) r = M.band(r, M.bnot(M.bxor(M.var(2 * i), M.var(2 * i + 1))));
  return r;
}

// make_and_circuit / make_or_circuit (and.rs:6-30, or.rs:6-30): bitwise op of two n-bit words, inputs a0 b0 a1 b1 ...
Fns build_bitwise(BddManager& M, uint32_t n, bool is_or) {
  Fns out(n);
  for (uint32_t i = 0; i < n; i++) out[i] = is_or ? M.bor(M.var(2 * i), M.var(2 * i + 1)) : M.band(M.var(2 * i), M.var(2 * i + 1));
  return out;
}

// bitshift (bitshift.rs:49-157): barrel shifter of 2:1 multiplexers.  Inputs are BIG-endian: variables
// 0..inputs are the value (index 0 = most significant bit), then shift_size shift-amount bits, most
// significant first; the low ceil(log2(inputs)) of them drive the stages, any higher one set clears the
// result (logical) or fills it with the sign (arithmetic).  mode: 0 logical, 1 rotation, 2 arithmetic.
Fns build_bitshift(BddManager& M, uint32_t inputs, uint32_t shift_size, bool right, uint32_t mode) {
  uint32_t used = 0;
  while ((1u << used) < inputs) used++;
  if (used == 0) used = 1;
  auto ite = [&](uint32_t c, uint32_t a, uint32_t b) { return M.bor(M.band(c, a), M.and_not(b, c)); };
  Fns result(inputs);
  for (uint32_t i = 0; i < inputs; i++) result[i] = M.var(i);
  const uint32_t old_msb = result[0];
  for (uint32_t i = 0; i < used; i++) {
    const uint32_t shift = 1u << (used - 1 - i);
    const uint32_t select = M.var(inputs + (shift_size - used) + i);
    const uint32_t k = shift % inputs;
    Fns inter(inputs);
    for (uint32_t j = 0; j < inputs; j++) inter[j] = right ? result[(j + inputs - k) % inputs] : result[(j + k) % inputs];
    Fns next(inputs);
    for (uint32_t j = 0; j < inputs; j++) {
      uint32_t shifted;
      if (mode == 0) shifted = (right ? j < shift : j + shift >= inputs) ? 0u : inter[j];
      else if (mode == 1) shifted = inter[j];
      else shifted = j < shift ? old_msb : inter[j];
      next[j] = ite(select, shifted, result[j]);
    }
    result.swap(next);
  }
  if (mode != 1) {
    uint32_t clear = 0;
    for (uint32_t x = 0; x < shift_size - used; x++) clear = M.bor(clear, M.var(inputs + x));
    const uint32_t fill = mode == 0 ? 0u : old_msb;
    for (uint32_t j = 0; j < inputs; j++) result[j] = ite(clear, fill, result[j]);
  }
  return result;
}

// mul_bdd_encode (mul.rs:149-179): the order in which the n*m (x, y) variable pairs appear, walking
// the anti-diagonals of the partial-product array from the most significant one; returns for every
// duplicated BDD variable the operand bit it stands for (x bits are 0..n, y bits n..n+m).
std::vector<uint32_t> multiplier_variable_map(uint32_t n, uint32_t m) {
  std::vector<uint32_t> enc;
  for (uint32_t d = n + m - 1; d >= 1; d--) {
    const uint32_t row = d > n ? d - n : 0, col = d > n ? 0 : n - d;
    for (uint32_t i = 0; row + i < m && col + i < n; i++) {
      enc.push_back(n - (col + i) - 1);  // x[n - c - 1]
      enc.push_back(n + row + i);        // y[r]
    }
  }
  return enc;
}

// multiplier_bdd (mul.rs:69-141) after Burch, "Using BDDs to Verify Multipliers": every cell of the
// m x n carry-save array gets its OWN copy of its x and y variable (2nm variables, ordered by
// mul_bdd_decode, mul.rs:183-221), which keeps every output BDD polynomial in size.
Fns build_multiplier(BddManager& M, uint32_t n, uint32_t m) {
  std::vector<uint32_t> x(n * m), y(n * m);
  auto idx = [n](uint32_t r, uint32_t c) { return r * n + c; };
  {
    uint32_t start_row = m - 1, start_col = n - 1, i = 0;
    for (;;) {
      for (uint32_t j = 0; j <= start_col && start_row + j < m; j++) {
        x[idx(start_row + j, start_col - j)] = M.var(i);
        y[idx(start_row + j, start_col - j)] = M.var(i + 1);
        i += 2;
      }
      if (start_row > 0) start_row--;
      else if (start_col > 0) start_col--;
      else break;
    }
  }
  std::vector<uint32_t> ands(n * m), sums(n * m, 0), carries(n * m, 0);
  for (uint32_t i = 0; i < n * m; i++) ands[i] = M.band(x[i], y[i]);
  for (uint32_t j = 0; j < n; j++) sums[j] = ands[idx(0, j)];
  for (uint32_t i = 1; i < m; i++)
    for (uint32_t j = 0; j < n; j++) {
      const uint32_t a = ands[idx(i, j)];
      const uint32_t b = j < n - 1 ? sums[idx(i - 1, j + 1)] : carries[idx(i - 1, j)];
      const uint32_t c_in = j > 0 ? carries[idx(i, j - 1)] : 0;
      const uint32_t axb = M.bxor(a, b);
      sums[idx(i, j)] = M.bxor(axb, c_in);
      carries[idx(i, j)] = M.bor(M.band(axb, c_in), M.band(b, a));
    }
  Fns result;
  for (uint32_t i = 0; i < m; i++) result.push_back(sums[idx(i, 0)]);
  for (uint32_t i = 1; i < n; i++) result.push_back(sums[idx(m - 1, i)]);
  result.push_back(carries[idx(m - 1, n - 1)]);
  return result;
}

// n_bits_are_true (mul.rs:227-251): exactly `k` of the operands are 1.  (The reference enumerates
// the combinations; the symmetric-function recurrence below gives the same Boolean function.)
uint32_t exactly_k(BddManager& M, const std::vector<uint32_t>& ops, uint32_t k) {
  std::vector<uint32_t> cnt(ops.size() + 2, 0);  // cnt[j]: exactly j of the operands seen so far are 1
  cnt[0] = 1;
  for (size_t i = 0; i < ops.size(); i++) {
    const uint32_t o = ops[i], no = M.bnot(o);
    for (size_t j = i + 1; j >= 1; j--) cnt[j] = M.bor(M.band(cnt[j], no), M.band(cnt[j - 1], o));
    cnt[0] = M.band(cnt[0], no);
  }
  return k <= ops.size() ? cnt[k] : 0;
}

void partition_integer(uint32_t n, uint32_t* lo, uint32_t* hi) {  // mul.rs:263-273, CIRCUIT_CUTOFF = 16
  if (n <= 16) { *lo = n; *hi = 0; return; }
  *hi = n / 2;
  *lo = n - n / 2;
}

// gradeschool_reduce_impl (mul.rs:428-586): sums the four shifted partial products of one
// divide-and-conquer step; input order is encode_gradeschool_reduction's (mul.rs:289-387).
Fns build_gradeschool_reduce(BddManager& M, uint32_t n, uint32_t m) {
  uint32_t a_lo, a_hi, b_lo, b_hi;
  partition_integer(n, &a_lo, &a_hi);
  partition_integer(m, &b_lo, &b_hi);
  Fns result(m + n, 0);
  uint32_t in = 0, out = 0, c0 = 0, c1 = 0, c2 = 0;
  for (uint32_t i = 0; i < b_lo; i++) result[i] = M.var(i);  // section 1: a_lo*b_lo passes through
  in += b_lo; out += b_lo;
  for (uint32_t i = 0; i < a_lo - b_lo; i++) {  // section 2: two summands
    const uint32_t a = M.var(in + 2 * i), b = M.var(in + 2 * i + 1);
    const std::vector<uint32_t> ops = {a, b, c0};
    result[out + i] = M.bxor(M.bxor(a, b), c0);
    c0 = M.bor(exactly_k(M, ops, 2), exactly_k(M, ops, 3));
  }
  in += 2 * (a_lo - b_lo); out += a_lo - b_lo;
  for (uint32_t i = 0; i < b_lo + b_hi; i++) {  // sections 3 and 4: three summands, two carries in
    const uint32_t a = M.var(in + 3 * i), b = M.var(in + 3 * i + 1), c = M.var(in + 3 * i + 2);
    const std::vector<uint32_t> ops = {a, b, c, c0, c1};
    result[out + i] = M.bxor(M.bxor(M.bxor(M.bxor(a, b), c), c0), c1);
    const uint32_t n0 = M.bor(exactly_k(M, ops, 2), exactly_k(M, ops, 3));
    const uint32_t n2 = M.bor(exactly_k(M, ops, 4), exactly_k(M, ops, 5));
    c0 = n0; c1 = c2; c2 = n2;
  }
  in += 3 * (b_lo + b_hi); out += b_lo + b_hi;
  for (uint32_t i = 0; i < a_hi - b_hi; i++) {  // section 5: two summands
    const uint32_t a = M.var(in + 2 * i), b = M.var(in + 2 * i + 1);
    const std::vector<uint32_t> ops = {a, b, c0, c1};
    result[out + i] = M.bxor(M.bxor(M.bxor(a, b), c0), c1);
    const uint32_t n0 = M.bor(exactly_k(M, ops, 2), exactly_k(M, ops, 3));
    const uint32_t n2 = exactly_k(M, ops, 4);
    c0 = n0; c1 = c2; c2 = n2;
  }
  in += 2 * (a_hi - b_hi); out += a_hi - b_hi;
  for (uint32_t i = 0; i < b_hi; i++) {  // section 6: carries ripple into a_hi*b_hi
    const uint32_t a = M.var(in + i);
    if (i <= 1) {
      const std::vector<uint32_t> ops = {a, c0, c1};
      result[out + i] = M.bxor(M.bxor(a, c0), c1);
      c0 = M.bor(exactly_k(M, ops, 2), exactly_k(M, ops, 3));
      if (i == 0) c1 = c2;
    } else {
      result[out + i] = M.bxor(a, c0);
      c0 = M.band(a, c0);
    }
  }
  return result;
}

// Multiplication by a plaintext constant k: the low n bits of x * k, inputs x0 .. x(n-1) least significant first, in
// their natural order (no duplicated copies as in build_multiplier), so output bit i is an ROBDD over x0 .. xi and
// every path tests each variable at most once: depth <= n.  The function is the ripple sum of the shifted copies
// x << j for every set bit j of k; its ROBDD is built directly from the states of that sum read least significant bit
// first instead of through apply() on the partial sums (which takes a minute at 32 bits):
// after x0 .. x(t-1), bit t + d of the product is bit d of C + k * (xt + 2 x(t+1) + ...), where the carry C =
// (k * (x0 .. x(t-1))) >> t < k matters only mod 2^(d+1).  Testing xt adds k * xt to C and shifts one bit out.
struct ConstMultiplier {
  BddManager& M;
  uint64_t k;
  std::unordered_map<uint64_t, uint32_t> memo;  // (t, d, C mod 2^(d+1)) -> BDD node
  uint32_t bit(uint32_t t, uint32_t d, uint64_t carry) {
    carry &= (2ull << d) - 1;  // d <= 31
    const uint64_t key = (uint64_t)t << 58 | (uint64_t)d << 52 | carry;
    auto it = memo.find(key);
    if (it != memo.end()) return it->second;
    const uint64_t lo = carry, hi = carry + k;
    const uint32_t r = d == 0 ? M.mk(t, (uint32_t)(lo & 1), (uint32_t)(hi & 1))
                              : M.mk(t, bit(t + 1, d - 1, lo >> 1), bit(t + 1, d - 1, hi >> 1));
    memo.emplace(key, r);
    return r;
  }
};

Fns build_const_multiplier(BddManager& M, uint32_t n, uint32_t k) {
  ConstMultiplier cm{M, k, {}};
  Fns out(n);
  for (uint32_t i = 0; i < n; i++) out[i] = cm.bit(0, i, 0);
  return out;
}

// ---- BDD -> multiplexer list ----------------------------------------------------------------------
// MuxCircuit::from(&[Bdd]) + remap_inputs + optimize (lib.rs:249-341,355-451): a BDD node testing
// variable v with children (lo, hi) is the multiplexer sel = input(v), low = lo, high = hi.  With a
// variable map (the multiplier) several BDD variables name the same input; re-hashing bottom-up on
// (input, low, high) merges what the renaming made equal -- the fixpoint of the reference's
// common_subexpression_elimination (opt.rs) -- and a multiplexer with low == high is its input.
int emit(BddManager& M, const Fns& outs, uint32_t n_inputs, const std::vector<uint32_t>* var_map, spf_mux_node** out, size_t* count) {
  if (M.overflow) return SPF_E_UNSUPPORTED;
  std::vector<uint8_t> live(M.nodes.size(), 0);
  {
    std::vector<uint32_t> stack(outs.begin(), outs.end());
    while (!stack.empty()) {
      const uint32_t v = stack.back();
      stack.pop_back();
      if (live[v]) continue;
      live[v] = 1;
      if (v > 1) { stack.push_back(M.nodes[v].lo); stack.push_back(M.nodes[v].hi); }
    }
  }
  std::vector<spf_mux_node> list;
  list.push_back({SPF_MUX_ZERO, 0, -1, -1, -1});
  list.push_back({SPF_MUX_ONE, 0, -1, -1, -1});
  for (uint32_t i = 0; i < n_inputs; i++) list.push_back({SPF_MUX_VARIABLE, i, -1, -1, -1});
  std::vector<int32_t> where(M.nodes.size(), -1);
  where[0] = 0;
  where[1] = 1;
  struct Key {
    uint32_t s, l, h;
    bool operator==(const Key& o) const { return s == o.s && l == o.l && h == o.h; }
  };
  struct KeyHash { size_t operator()(const Key& k) const { return (size_t)BddManager::mix(k.s, k.l, k.h); } };
  std::unordered_map<Key, int32_t, KeyHash> seen;
  for (uint32_t v = 2; v < M.nodes.size(); v++) {  // ids ascend from children to parents
    if (!live[v]) continue;
    const uint32_t input = var_map ? (*var_map)[M.nodes[v].var] : M.nodes[v].var;
    const int32_t lo = where[M.nodes[v].lo], hi = where[M.nodes[v].hi];
    if (lo == hi) { where[v] = lo; continue; }
    const Key k{input, (uint32_t)lo, (uint32_t)hi};
    auto it = seen.find(k);
    if (it != seen.end()) { where[v] = it->second; continue; }
    where[v] = (int32_t)list.size();
    seen.emplace(k, where[v]);
    list.push_back({SPF_MUX_MUX, 0, (int32_t)(2 + input), lo, hi});
  }
  for (size_t i = 0; i < outs.size(); i++) list.push_back({SPF_MUX_OUTPUT, (uint32_t)i, -1, where[outs[i]], -1});
  spf_mux_node* buf = static_cast<spf_mux_node*>(malloc(list.size() * sizeof(spf_mux_node)));
  if (!buf) return SPF_E_INVALID;
  memcpy(buf, list.data(), list.size() * sizeof(spf_mux_node));
  *out = buf;
  *count = list.size();
  return SPF_OK;
}

}  // namespace

extern "C" {

static int mux_circuit_impl(uint32_t kind, uint32_t n, uint32_t m, uint32_t flags, spf_mux_node** out, size_t* count);
int spf_b200_mux_circuit(uint32_t kind, uint32_t n, uint32_t m, uint32_t flags, spf_mux_node** out, size_t* count) {
  try {  // C++ exceptions (std::bad_alloc on a huge BDD) never cross the C ABI
    return mux_circuit_impl(kind, n, m, flags, out, count);
  } catch (...) {
    return SPF_E_INVALID;
  }
}
static int mux_circuit_impl(uint32_t kind, uint32_t n, uint32_t m, uint32_t flags, spf_mux_node** out, size_t* count) {
  if (!out || !count) return SPF_E_INVALID;
  *out = nullptr;
  *count = 0;
  const bool f0 = flags & 1, f1 = flags & 2;
  if (n == 0 || n > 4096 || m > 4096) return SPF_E_INVALID;
  switch (kind) {
    case SPF_MUX_RIPPLE_CARRY_ADDER: {
      if (m == 0) return SPF_E_INVALID;
      BddManager M(n + m + (f0 ? 1 : 0));
      return emit(M, build_adder(M, n, m, f0), M.nvars, nullptr, out, count);
    }
    case SPF_MUX_FULL_SUBTRACTOR: {
      BddManager M(2 * n + (f0 ? 1 : 0));
      return emit(M, build_subtractor(M, n, f0), M.nvars, nullptr, out, count);
    }
    case SPF_MUX_NEGATOR: {
      BddManager M(n);
      return emit(M, build_negator(M, n), n, nullptr, out, count);
    }
    case SPF_MUX_COMPARE: {
      BddManager M(2 * n);
      return emit(M, Fns{unsigned_compare(M, n, f0, f1)}, 2 * n, nullptr, out, count);
    }
    case SPF_MUX_COMPARE_SIGNED: {
      BddManager M(2 * n);
      return emit(M, Fns{signed_compare(M, n, f0, f1)}, 2 * n, nullptr, out, count);
    }
    case SPF_MUX_COMPARE_EQUAL: {
      BddManager M(2 * n);
      const uint32_t eq = all_pairs_equal(M, n);
      return emit(M, Fns{f0 ? M.bnot(eq) : eq}, 2 * n, nullptr, out, count);
    }
    case SPF_MUX_BITWISE: {
      BddManager M(2 * n);
      return emit(M, build_bitwise(M, n, f0), 2 * n, nullptr, out, count);
    }
    case SPF_MUX_BITSHIFT: {  // n = value width, m = shift-amount width; flags bit0 = right, bits 1-2 = mode
      const uint32_t mode = (flags >> 1) & 3;
      uint32_t used = 0;
      while ((1u << used) < n) used++;
      if (used == 0) used = 1;
      if (m < used || mode > 2) return SPF_E_INVALID;                       // bitshift.rs:57-60
      if (mode == 1 && (n & (n - 1)) != 0) return SPF_E_INVALID;            // rotation: power-of-two widths only (:64-66)
      if (mode == 2 && !f0) return SPF_E_INVALID;                           // arithmetic shifts are right shifts (:68-70)
      BddManager M(n + m);
      return emit(M, build_bitshift(M, n, m, f0, mode), n + m, nullptr, out, count);
    }
    case SPF_MUX_UNSIGNED_MULTIPLIER: {
      if (m == 0 || (uint64_t)n * m * 2 >= (1u << 16)) return SPF_E_INVALID;  // mul.rs:36 (u16 variable ids)
      if ((uint64_t)n * m * 2 > 16384) return SPF_E_UNSUPPORTED;  // apply() recurses once per variable: bound the stack
      BddManager M(2 * n * m);
      const Fns f = build_multiplier(M, n, m);
      const std::vector<uint32_t> map = multiplier_variable_map(n, m);
      return emit(M, f, n + m, &map, out, count);
    }
    case SPF_MUX_GRADESCHOOL_REDUCE: {
      if (m == 0 || n < m) return SPF_E_INVALID;  // mul.rs:431
      BddManager M(2 * (n + m));
      return emit(M, build_gradeschool_reduce(M, n, m), 2 * (n + m), nullptr, out, count);
    }
    case SPF_MUX_CONST_MULTIPLIER: {  // n input bits, flags = the constant (its low n bits count)
      if (n > 32 || m != 0) return SPF_E_INVALID;
      BddManager M(n);
      return emit(M, build_const_multiplier(M, n, n == 32 ? flags : flags & ((1u << n) - 1)), n, nullptr, out, count);
    }
    default:
      return SPF_E_INVALID;
  }
}

void spf_b200_mux_free(spf_mux_node* nodes) { free(nodes); }

}  // extern "C"
