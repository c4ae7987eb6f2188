// Device-side building blocks of the tree store (hmz_tree.cu).
//
// A search is owned by a PAIR of lanes (16 searches per warp).  Lane h of the pair owns half h of
// every 128-byte node record: the three 16-byte child slots 3h..3h+2 and their priors, i.e. four
// 128-bit loads of 64 contiguous bytes, evaluated with 3-way instruction-level parallelism; one
// shuffle merges the two lanes' candidates.  Why pairs: ncu / clock timelines of the earlier forms
// showed (a) 8 lanes per search (one child per lane, shuffle arg-max) issue-bound — ~36 warp
// instructions per search-level, a quarter of the lanes idle; (b) one thread per search bound by
// the L1 tag stage, which serves one 128-byte line per cycle: 8 x LDG.128 with 32 different lines
// each = 256 cycles per warp-level.  Pairs need ~14 instructions and 4 line-cycles per search-level.
//
// Arithmetic contract (bit-exact vs the reference, SURVEY.md §8a a14-a19):
//   Q, W, value, min/max  : IEEE float64, every op an explicit __d*_rn so nvcc cannot contract
//                           the reference's separate multiply and add into an FMA;
//   f32(Q) + f32(U)       : float32 add after rounding each term (MCTS/node.py:83,103,123);
//   U = prior * w         : float32 x float32 for a float32 prior (NumPy >= 2 weak scalars),
//                           float64 product then rounded at a Dirichlet-noised root (:122);
//   ties                  : lowest action index (the sanctioned replacement of :86).
#pragma once
#include <type_traits>
#include <math.h>

#include "hmz_common.cuh"

namespace hmz {

static_assert(sizeof(hmz_child_t) == 16 && sizeof(hmz_half_t) == 64 && sizeof(hmz_node_t) == 128,
              "node record layout (include/hmz.h) must be 2 x 64-byte halves of 3 x 16-byte child slots");

// Host: validates a search descriptor and makes sure the per-device constant tables / kernel attributes are in place.
int check_search(const hmz_search_t* s, const char* who);

constexpr int kPathCap = 32;  // path levels recorded for the backup (deeper paths walk parent links)

// Tooling: clock64() marks of one lane pair (hmz_debug_tree_timeline), compiled only into the kTL = true
// instantiations.  `dep` makes the clock read wait for a loaded value.
static __device__ unsigned long long g_tree_timeline[64];
static __device__ long long g_tree_timeline_search = -1;
template <bool kTL>
__device__ __forceinline__ void tree_mark(int slot, bool on, uint32_t dep = 0u) {
  if (kTL && on && dep != 0xFFFFFFF1u) g_tree_timeline[slot] = clock64();
}

struct Leaf {
  int parent;  // record of the leaf's parent
  int action;  // action from that parent to the (unexpanded) leaf
  int depth;   // number of best_child steps taken (>= 1)
};

// 16-byte child slot <-> registers
struct Slot {
  double W;
  float rwd;
  int n, child;
  __device__ __forceinline__ static Slot unpack(const uint4& q) {
    Slot s;
    s.W = __hiloint2double((int)q.y, (int)q.x);
    s.rwd = __uint_as_float(q.z);
    s.n = (int)(q.w & 0xFFFFu);
    s.child = (int)(q.w >> 16);
    return s;
  }
  __device__ __forceinline__ uint4 pack() const {
    return make_uint4((uint32_t)__double2loint(W), (uint32_t)__double2hiint(W), __float_as_uint(rwd),
                      (uint32_t)n | ((uint32_t)child << 16));
  }
};

// 256-bit global accesses (sm_100: LDG.256 / STG.256): half a node record in two instructions
__device__ __forceinline__ void ld256(const void* p, uint4& lo, uint4& hi) {
  asm volatile("ld.global.v8.u32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(lo.x), "=r"(lo.y), "=r"(lo.z), "=r"(lo.w), "=r"(hi.x), "=r"(hi.y), "=r"(hi.z), "=r"(hi.w)
               : "l"(p)
               : "memory");
}
__device__ __forceinline__ void st256(void* p, const uint4& lo, const uint4& hi) {
  asm volatile("st.global.v8.u32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "r"(lo.x), "r"(lo.y), "r"(lo.z), "r"(lo.w),
               "r"(hi.x), "r"(hi.y), "r"(hi.z), "r"(hi.w)
               : "memory");
}

__device__ __forceinline__ uint4* slot_ptr(hmz_node_t* nodes, int e, int a) {
  return reinterpret_cast<uint4*>(&nodes[e].h[a / 3].c[a % 3]);
}

// Node.expand (MCTS/node.py:30-51) of a fresh node: six children with priors `pr`, N = 0, W = 0,
// rwd = 0, no expanded grandchildren.  Lane `half` of the pair writes its 64-byte half.
__device__ __forceinline__ void write_fresh_half_vals(hmz_node_t* rec, int half, float pr0, float pr1, float pr2, int parent,
                                                      int parent_action) {
  uint4* dst = reinterpret_cast<uint4*>(&rec->h[half]);
  const uint4 empty = make_uint4(0u, 0u, 0u, 0xFFFF0000u);  // W = 0, rwd = 0, N = 0, child = HMZ_NO_CHILD
  st256(dst, empty, empty);
  st256(dst + 2, empty,
        make_uint4(__float_as_uint(pr0), __float_as_uint(pr1), __float_as_uint(pr2),
                   half == 0 ? ((uint32_t)parent | ((uint32_t)parent_action << 16)) : 0u));
}
__device__ __forceinline__ void write_fresh_half(hmz_node_t* rec, int half, const float* __restrict__ pr, int parent,
                                                 int parent_action) {
  write_fresh_half_vals(rec, half, pr[3 * half], pr[3 * half + 1], pr[3 * half + 2], parent, parent_action);
}
// A float the network kernel wrote: through the read-only path when that kernel has COMPLETED before this one reads
// (stand-alone launches), a plain coherent load when it is written by other CTAs of the same kernel (persistent schedule).
template <bool kReadOnly>
__device__ __forceinline__ float ld_net_out(const float* p) {
  return kReadOnly ? __ldg(p) : *p;
}

// ---- exact float64 division without the generic division routine ---------------------------------
// The reference divides by small integers (visit counts, N + 1) and by the min-max range.  For a
// positive divisor b whose correctly rounded reciprocal y = RN(1/b) is known — a host-computed table for
// integers, one __drcp_rn per search and launch for the range — two Markstein corrections
//     q0 = RN(a y);  r0 = a - b q0 (exact, one FMA);  q1 = RN(q0 + r0 y);  r1 = a - b q1;  q = RN(q1 + r1 y)
// give the correctly rounded quotient RN(a / b): q1 is within half an ulp (+ 2^-53 ulp) of a / b, i.e.
// faithful, and Markstein's theorem (Markstein 1990; Cornea, Harrison, Tang 2002, thm. on FMA-based
// division) then makes the second correction exact for every b whose significand is not all ones.
// Operands outside the comfortably normal range (and b with an all-ones significand) take __ddiv_rn.
// tests/test_div_gpu.py compares this bit for bit with __ddiv_rn on ~10^9 operand pairs.
constexpr int kRcpTable = 4096;
static __device__ double g_rcp[kRcpTable + 1];  // g_rcp[k] = RN(1 / k) for k >= 1 (filled by the host, IEEE division)

// The walk needs, per child with visit count n: 1/max(n,1), 1/(n+1) and both divisors as doubles.  One 32-byte row
// per count replaces two clamps, two table loads and two int -> float64 conversions.
struct __align__(32) CountRow {
  double rcp_n, rcp_n1, dn, dn1;  // 1/max(n,1), 1/(n+1), (double)max(n,1), (double)(n+1)
};
static __device__ CountRow g_cnt[kRcpTable];  // n in [0, kRcpTable): n + 1 <= kRcpTable

// Where the walk and the backup read their constant tables from.  GlobalTables: the __device__ arrays above through the
// read-only path (stand-alone kernels: L1-resident).  SmemTables: a shared-memory copy of the first `rows` count rows
// and of the pUCT table — the persistent kernel's tree CTAs acquire at every hand-off, which invalidates L1, so global
// tables would cost an L2 round trip per dependent lookup; `rows` must exceed every visit count of the search.
struct GlobalTables {
  __device__ __forceinline__ double rcp(int n) const { return __ldg(&g_rcp[min(n, kRcpTable)]); }
  __device__ __forceinline__ void count_row(int n, double2& lo, double2& hi) const {
    const double2* row = reinterpret_cast<const double2*>(&g_cnt[min(n, kRcpTable - 1)]);
    lo = __ldg(row);
    hi = __ldg(row + 1);
  }
  __device__ __forceinline__ double ucb(const double* __restrict__ ucb_table, int n) const { return ucb_table[n]; }
};
struct SmemTables {
  const CountRow* cnt;  // shared memory, `rows` rows
  const double* ucb_s;  // shared memory, `rows` entries
  int rows;
  __device__ __forceinline__ double rcp(int n) const { return cnt[min(n, rows - 1)].rcp_n; }  // 1 / n for n >= 1
  __device__ __forceinline__ void count_row(int n, double2& lo, double2& hi) const {
    const double2* row = reinterpret_cast<const double2*>(&cnt[min(n, rows - 1)]);
    lo = row[0];
    hi = row[1];
  }
  __device__ __forceinline__ double ucb(const double* __restrict__, int n) const { return ucb_s[min(n, rows - 1)]; }
};

// |a| comfortably normal (2^-830 <= |a| < 2^830), tested on the exponent bits with integer instructions
__device__ __forceinline__ bool div_fast_ok(double a) {
  const unsigned hi = (unsigned)__double2hiint(a) & 0x7FFFFFFFu;
  return (hi - 0x0C100000u) < (0x73D00000u - 0x0C100000u);
}
__device__ __forceinline__ double div_refine(double a, double b, double y) {
  double q = __dmul_rn(a, y);
  double r = __fma_rn(-b, q, a);
  q = __fma_rn(r, y, q);
  r = __fma_rn(-b, q, a);
  return __fma_rn(r, y, q);
}
// An operand the two-correction division handles exactly: +0 or comfortably normal.
__device__ __forceinline__ bool div_operand_ok(double a) {
  return (__double_as_longlong(a) == 0ll) | div_fast_ok(a);
}
// "Tame": +-0 or 2^-700 <= |a| < 2^700 (NaN / Inf are not).  The fused hot loop keeps a sticky per-search flag
// "some W or Q written by a backup was not tame" instead of testing every operand of every walk: if all W and all
//   Q = rwd + discount * W / N  (every one of which also went through the min/max update, so mn <= Q <= mx)
// are tame, then W is a valid operand of the two-correction division, and so is  num = Q - mn:  0 <= num <=
// mx - mn < 2^701, and a nonzero difference of two tame doubles is at least 2^-700 * 2^-52 > 2^-830.
__device__ __forceinline__ bool is_tame(double a) {
  const unsigned hi = (unsigned)__double2hiint(a) & 0x7FFFFFFFu;
  return (__double_as_longlong(a) == 0ll) | ((hi - 0x14300000u) < (0x6BB00000u - 0x14300000u));
}
// a / n for a visit count n >= 1: the shortcut is evaluated unconditionally (straight-line code), the rare
// operand outside its proven range takes the generic division afterwards
template <class TB>
__device__ __forceinline__ double div_by_count(double a, int n, const TB& tb) {
  const double q = div_refine(a, (double)n, tb.rcp(n));
  if ((n > kRcpTable) | !div_operand_ok(a)) return __ddiv_rn(a, (double)n);
  return q;
}
__device__ __forceinline__ double div_by_count(double a, int n) { return div_by_count(a, n, GlobalTables()); }
// a / b with y = __drcp_rn(b) precomputed; y_ok = b is positive, comfortably normal and its significand is not all ones
__device__ __forceinline__ double div_by_known(double a, double b, double y, bool y_ok) {
  if (y_ok && div_fast_ok(a)) return div_refine(a, b, y);
  return __ddiv_rn(a, b);
}
__device__ __forceinline__ bool rcp_usable(double b) {
  const unsigned long long bits = (unsigned long long)__double_as_longlong(b);
  return (b > 0.0) & div_fast_ok(b) & ((bits & 0xFFFFFFFFFFFFFull) != 0xFFFFFFFFFFFFFull);
}

__device__ __forceinline__ void minmax_update(double x, double& mn, double& mx) {
  if (x > mx) mx = x;  // python max(maximum, value): value only when strictly greater
  if (x < mn) mn = x;
}

// Reference-order evaluation of one child (the slow, always-exact form): used when an operand falls
// outside the range the straight-line form below is proven for.
static __device__ __noinline__ float child_score_exact(double W, float rwd, int n, float prior, double prior64, bool use64, double tn,
                                                double discount, double mn, double range, bool normalise) {
  float qf = 0.0f;  // child_Q: 0 for unvisited children (node.py:98-102)
  if (n > 0) {
    double q = __dadd_rn((double)rwd, __dmul_rn(discount, __ddiv_rn(W, (double)n)));
    if (normalise) q = __ddiv_rn(__dsub_rn(q, mn), range);
    qf = __double2float_rn(q);
  }
  const double w = __ddiv_rn(tn, (double)(n + 1));
  const float u = use64 ? __double2float_rn(__dmul_rn(prior64, w)) : __fmul_rn(prior, __double2float_rn(w));
  return __fadd_rn(qf, u);
}

// Node.best_child repeated from the root until an unexpanded child (MCTS/mcts.py:80-86,
// MCTS/node.py:72-123), for the pair of lanes that owns the search (`half` = lane & 1).
//   root_n        root.N  (= number of completed simulations)
//   root_prior64  float64 root priors when the root was Dirichlet-noised, else nullptr
//   path_out      nullable [path_cap] bytes: chosen action per level (diagnostics)
//   path_elem     nullable [kPathCap] 32-byte elements, one per level, for the next backup: the chosen child's
//                 16-byte slot AS READ HERE (nothing touches the tree until that backup) and the word
//                 (record | action << 16) — so the backup needs no second, dependent round trip for the slots
// The three children of a lane are evaluated as ONE straight-line block (no data-dependent branch
// between them), so their float64 chains interleave: every division is the two-correction form of
// div_refine on reciprocals fetched up front, unvisited children are computed and discarded, and the
// rare operand outside the proven range re-evaluates the lane's children with child_score_exact.
// The loop is WARP-UNIFORM: every lane stays in it until the deepest of the warp's 16 walks has ended
// (`active` masks the memory accesses of finished or out-of-range pairs), so the pair exchange is a plain
// full-mask shuffle — a pair-masked shuffle inside a divergent loop costs a MATCH/REDUX/VOTE sequence per
// call — and the walk needs no reconvergence bookkeeping.  ALL 32 lanes of the warp must call it.
//   kTrusted / wild   hot loop only: the per-operand range tests are replaced by `wild` (the search's sticky flag or
//                     untame persisted bounds) plus a per-launch test of the largest possible count; see is_tame()
template <bool kTL = false, bool kTrusted = false, class TB = GlobalTables>
__device__ __forceinline__ Leaf select_leaf(const hmz_node_t* nodes, const double* __restrict__ root_prior64, double mn,
                                            double mx, int root_n, const double* __restrict__ ucb_table,
                                            double discount, int half, uint8_t* __restrict__ path_out, int path_cap,
                                            uint4* __restrict__ path_elem, bool tl_on = false, bool active = true,
                                            bool wild = false, const TB& tb = TB()) {
  const bool normalise = mx > mn;  // MinMaxStats.normalize (MCTS/utils_mcts.py:12-16)
  const double range = __dsub_rn(mx, mn);
  const bool range_ok = normalise & rcp_usable(range);
  const double range_rcp = range_ok ? __drcp_rn(range) : 0.0;
  // trusted mode: every count on the walk is <= root_n, the bounds persist from earlier searches (test them here)
  const bool distrust = wild | (root_n + 1 > kRcpTable) | (normalise & (!range_ok | !is_tame(mn) | !is_tame(mx)));
  int e = 0, n_parent = root_n, depth = 0;
  Leaf leaf{0, 0, 0};
  uint4 q0 = make_uint4(0u, 0u, 0u, 0xFFFF0000u), q1 = q0, q2 = q0, q3 = make_uint4(0u, 0u, 0u, 0u);
  // One level of the walk.  The level body exists twice: the first level of a search whose root priors are float64
  // (Dirichlet-noised) and every other level, which then carries none of the float64-prior work.
  auto level = [&](auto root64_tag) {
    constexpr bool kRoot64 = decltype(root64_tag)::value;
    const bool use64 = kRoot64 && (e == 0) & (root_prior64 != nullptr);
    double rp64[3] = {0.0, 0.0, 0.0};
    double tn = 0.0;
    if (active) {
      const uint4* hp = reinterpret_cast<const uint4*>(&nodes[e].h[half]);
      ld256(hp, q0, q1);
      ld256(hp + 2, q2, q3);
      if (depth == 0) tree_mark<kTL>(41, tl_on);
      tn = tb.ucb(ucb_table, n_parent);
      if (use64) {  // only the (noised) root has float64 priors; requested together with the record
#pragma unroll
        for (int j = 0; j < 3; ++j) rp64[j] = root_prior64[3 * half + j];
      }
    }
    if (depth < 8) tree_mark<kTL>(8 + 2 * depth, tl_on, q0.w ^ q1.w ^ q2.w ^ q3.w);
    Slot c[3] = {Slot::unpack(q0), Slot::unpack(q1), Slot::unpack(q2)};
    const float prior[3] = {__uint_as_float(q3.x), __uint_as_float(q3.y), __uint_as_float(q3.z)};
    double y[3], yw[3], dn[3], dn1[3];
#pragma unroll
    for (int j = 0; j < 3; ++j) {  // reciprocals first: independent L1 hits
      // counts beyond the table are flagged below (their results are discarded), so the clamp only keeps the load in range
      double2 lo, hi;
      tb.count_row(c[j].n, lo, hi);
      y[j] = lo.x;
      yw[j] = lo.y;
      dn[j] = hi.x;
      dn1[j] = hi.y;
    }
    float score[3];
    bool exact_needed = !div_operand_ok(tn) | (kTrusted & distrust);
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      const int n = c[j].n;
      const double t1 = div_refine(c[j].W, dn[j], y[j]);
      const double q = __dadd_rn((double)c[j].rwd, __dmul_rn(discount, t1));
      const double num = __dsub_rn(q, mn);
      const double qn = normalise ? div_refine(num, range, range_rcp) : q;
      const float qf = n > 0 ? __double2float_rn(qn) : 0.0f;  // child_Q: 0 for unvisited children (node.py:98-102)
      // child_U: w = (log((N+c_base+1)/c_base) + c_init) * sqrt(N) / (child.N + 1)  (node.py:114-121)
      const double w = div_refine(tn, dn1[j], yw[j]);
      // float64 prior (noised root): product in float64; float32 prior: weak scalar -> float32 product (node.py:122)
      const float u = use64 ? __double2float_rn(__dmul_rn(rp64[j], w)) : __fmul_rn(prior[j], __double2float_rn(w));
      score[j] = __fadd_rn(qf, u);  // node.py:83 on float32 arrays
      // bitwise, not short-circuit: a data-dependent branch here would fence the three children's chains apart
      if (!kTrusted)
        exact_needed |= (n + 1 > kRcpTable) |
                        ((n > 0) & (!div_operand_ok(c[j].W) | (normalise & (!range_ok | !div_operand_ok(num)))));
    }
    if (exact_needed & active) {
#pragma unroll
      for (int j = 0; j < 3; ++j)
        score[j] = child_score_exact(c[j].W, c[j].rwd, c[j].n, prior[j], rp64[j], use64, tn, discount, mn, range, normalise);
    }
    float best_score = score[0];
    int best = 3 * half, best_child = c[0].child, best_n = c[0].n;
#pragma unroll
    for (int j = 1; j < 3; ++j)
      if (score[j] > best_score) {  // first maximum wins inside the half
        best_score = score[j];
        best = 3 * half + j;
        best_child = c[j].child;
        best_n = c[j].n;
      }
    // merge the two halves: actions 0..2 (lane 0) beat 3..5 (lane 1) on equal scores
    const float other_score = __shfl_xor_sync(0xffffffffu, best_score, 1);
    const int other_pack = __shfl_xor_sync(0xffffffffu, best | (best_child << 16), 1);
    const int other_n = __shfl_xor_sync(0xffffffffu, best_n, 1);
    const bool take_other = half == 0 ? (other_score > best_score) : !(best_score > other_score);
    if (take_other) {
      best = other_pack & 7;
      best_child = (int)((unsigned)other_pack >> 16);
      best_n = other_n;
    }
    if (active) {
      if (half == 0) {
        if (path_out != nullptr && depth < path_cap) path_out[depth] = (uint8_t)best;
      }
      if (path_elem != nullptr && depth < kPathCap && (best >= 3) == (half == 1)) {  // the lane that holds the chosen slot
        const int j = best - 3 * half;
        const uint4 qs = j == 0 ? q0 : (j == 1 ? q1 : q2);
        st256(path_elem + 2 * depth, qs, make_uint4((uint32_t)e | ((uint32_t)best << 16), 0u, 0u, 0u));
      }
      if (depth < 8) tree_mark<kTL>(9 + 2 * depth, tl_on, (uint32_t)best_child);
      ++depth;
      if (best_child == (int)HMZ_NO_CHILD) {
        leaf.parent = e;
        leaf.action = best;
        leaf.depth = depth;
        active = false;
      } else {
        e = best_child;
        n_parent = best_n;
      }
    }
  };
  bool first = true;
  while (__any_sync(0xffffffffu, active)) {
    if (first && root_prior64 != nullptr)  // uniform: every lane is at its root in the first iteration
      level(std::true_type{});
    else
      level(std::false_type{});
    first = false;
  }
  return leaf;
}

// node.expand bookkeeping on the parent slot + Node.backup (MCTS/node.py:53-70) from the leaf to
// the root by walking parent links (any depth).  `value` enters as the network value of the new node.
template <class TB = GlobalTables>
__device__ __forceinline__ void backup_walk(hmz_node_t* nodes, int pe, int pa, int sim, float r, double value,
                                            double discount, double& root_w, double& mn, double& mx, bool& wild,
                                            const TB& tb = TB()) {
  int e = pe, a = pa;
  bool leaf = true;
  while (true) {
    uint4* sp = slot_ptr(nodes, e, a);
    Slot c = Slot::unpack(*sp);
    if (leaf) {  // leaf.rwd = reward, the leaf is now the expanded record sim + 1 (node.py:44-49)
      c.rwd = r;
      c.child = sim + 1;
      leaf = false;
    }
    c.W = __dadd_rn(c.W, value);  // current.W += value
    c.n += 1;                     // current.N += 1
    *sp = c.pack();
    const double rwd = (double)c.rwd;
    const double qv = __dadd_rn(rwd, __dmul_rn(discount, div_by_count(c.W, c.n, tb)));
    wild |= !is_tame(c.W) | !is_tame(qv);
    minmax_update(qv, mn, mx);
    value = __dadd_rn(rwd, __dmul_rn(discount, value));  // value = rwd + discount * value
    if (e == 0) break;
    a = nodes[e].h[0].parent_action;
    e = nodes[e].h[0].parent;
  }
  // the root itself: rwd = 0.0 (MCTS/mcts.py:69), N = sim + 1 after this backup
  root_w = __dadd_rn(root_w, value);
  const double q_root = __dadd_rn(0.0, __dmul_rn(discount, div_by_count(root_w, sim + 1, tb)));
  wild |= !is_tame(q_root);
  minmax_update(q_root, mn, mx);
}

// Same backup for a path of depth <= kPathCap recorded by select_leaf as 32-byte path elements (slot + entry), four
// levels per batch.  A batch is loaded with four independent 256-bit loads from consecutive addresses that depend
// only on the search index, then the leaf-to-root float64 recurrence runs in registers and the updated slots are
// stored to their home records.  Operation for operation identical to backup_walk, so results are bit-identical.
struct PathBatch {
  uint4 slot[4];
  uint32_t ent[4];
};

__device__ __forceinline__ void load_batch4(const uint4* __restrict__ path_elem, int k0, int depth, PathBatch& pb) {
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    uint4 meta = make_uint4(0u, 0u, 0u, 0u);
    if (k0 + j < depth) ld256(path_elem + 2 * (k0 + j), pb.slot[j], meta);
    pb.ent[j] = meta.x;
  }
}

template <class TB = GlobalTables>
__device__ __forceinline__ void backup_batch4(hmz_node_t* nodes, const PathBatch& pb, int k0, int depth, int sim, float r,
                                              double& value, double discount, double& mn, double& mx, bool& wild,
                                              const TB& tb = TB()) {
#pragma unroll
  for (int j = 3; j >= 0; --j) {
    if (k0 + j < depth) {
      Slot c = Slot::unpack(pb.slot[j]);
      if (k0 + j == depth - 1) {  // the leaf slot: Node.expand bookkeeping on the parent (node.py:44-49)
        c.rwd = r;
        c.child = sim + 1;
      }
      c.W = __dadd_rn(c.W, value);  // current.W += value
      c.n += 1;                     // current.N += 1
      *slot_ptr(nodes, (int)(pb.ent[j] & 0xFFFFu), (int)(pb.ent[j] >> 16)) = c.pack();
      const double rwd = (double)c.rwd;
      const double qv = __dadd_rn(rwd, __dmul_rn(discount, div_by_count(c.W, c.n, tb)));
      wild |= !is_tame(c.W) | !is_tame(qv);
      minmax_update(qv, mn, mx);
      value = __dadd_rn(rwd, __dmul_rn(discount, value));  // value = rwd + discount * value
    }
  }
}

// Levels >= 4, leaf side first (lane 1 of the pair): `pb` holds the leaf-side batch k_top = (depth - 1) & ~3 >= 4.
template <class TB = GlobalTables>
__device__ __forceinline__ void backup_deep(hmz_node_t* nodes, const uint4* __restrict__ path_elem, PathBatch& pb, int depth, int sim,
                                            float r, double& value, double discount, double& mn, double& mx, bool& wild,
                                            const TB& tb = TB()) {
#pragma unroll 1
  for (int k0 = (depth - 1) & ~3; k0 >= 4; k0 -= 4) {
    backup_batch4(nodes, pb, k0, depth, sim, r, value, discount, mn, mx, wild, tb);
    if (k0 >= 8) load_batch4(path_elem, k0 - 4, depth, pb);
  }
}

// Levels 0..3 and the root itself (lane 0 of the pair): rwd = 0.0 at the root (MCTS/mcts.py:69), N = sim + 1 after this backup.
template <class TB = GlobalTables>
__device__ __forceinline__ void backup_top(hmz_node_t* nodes, const PathBatch& pb, int depth, int sim, float r, double value,
                                           double discount, double& root_w, double& mn, double& mx, bool& wild,
                                           const TB& tb = TB()) {
  backup_batch4(nodes, pb, 0, depth, sim, r, value, discount, mn, mx, wild, tb);
  root_w = __dadd_rn(root_w, value);
  const double q_root = __dadd_rn(0.0, __dmul_rn(discount, div_by_count(root_w, sim + 1, tb)));
  wild |= !is_tame(q_root);
  minmax_update(q_root, mn, mx);
}

// Scratch of hmz_search_run per search (hmz_search_workspace_bytes): the leaf of the pending simulation, the path
// elements its walk recorded, the sticky tameness flag, and the network outputs of that simulation.
struct TreeScratch {
  uint16_t* leaf_parent;
  uint8_t* leaf_action;
  uint16_t* leaf_depth;
  uint4* path_elem;
  uint8_t* wild_flags;
  const float* r;
  const float* p;
  const float* v;
  float* capture;  // nullable: [n_searches][8] row of THIS simulation
  unsigned long long* gantt;  // tooling (hmz_debug_gantt), nullable
  const uint16_t* budget;     // nullable: simulations of each search (hmz_search_run_multi); the search backs up simulation
                              // sim only if sim < budget and selects for sim + 1 only if sim + 1 < budget
};

// Hand-off words of the server schedule (hmz_persist.cu), one 32-byte sector per 256-search tile pair each.
struct ServerCtl {
  uint32_t* tree_done;  // warps that have finished the pair's selections: 16 per simulation
  uint32_t* mlp_done;   // simulations whose network outputs are complete for the pair
  uint32_t* group_done; // (one sector per stream group) passes the network CTAs have finished for the group's pairs
};

// Phases 2b + 3 of simulation `sim` (expansion with the network outputs, backup), optionally followed at once by the
// selection of simulation `sim + 1` — the fused hot-loop form: the path just updated is still close and the next walk
// usually shares its prefix.  With path elements (slot + entry per level, recorded by the previous walk) the backup needs
// one round trip for its inputs; without them (split-phase API) it walks the parent links.
//   b_raw, half   the search this lane pair owns (b_raw >= n_searches: masked, but the lane stays for the warp-uniform walk)
//   do_select     bit 0: select simulation sim + 1 afterwards; bit 4: no backup (with sim = -1: the first selection
//                 of a search)
//   kTrusted      `wild_flags[search]` is the sticky "a backup wrote an untame W or Q" flag of is_tame(); the walk then
//                 skips its per-operand range tests
//   kPdl          stand-alone kernel launched as a programmatic dependent of the network kernel: it signals its own
//                 dependents at entry and waits for the network kernel after loading what the previous tree kernel wrote
// ALL 32 lanes of the warp must call it.
template <bool kTL, bool kTrusted, bool kPdl, class TB>
__device__ __forceinline__ void tree_phase(const hmz_search_t& s, int sim, const double* __restrict__ ucb_table, double discount,
                                           const TreeScratch& sc, int do_select, int64_t b_raw, int half, const TB& tb) {
  uint16_t* leaf_parent = sc.leaf_parent;
  uint8_t* leaf_action = sc.leaf_action;
  uint16_t* leaf_depth = sc.leaf_depth;
  uint4* path_elem = sc.path_elem;
  uint8_t* wild_flags = sc.wild_flags;
  const float* r = sc.r;
  const float* p = sc.p;
  const float* v = sc.v;
  float* capture = sc.capture;
  if (kPdl) pdl_launch_dependents();
  const bool valid = b_raw < s.n_searches;  // out-of-range pairs stay for the warp-uniform walk, masked
  const int64_t b = valid ? b_raw : s.n_searches - 1;
  const bool tl = kTL && valid && b == (g_tree_timeline_search & 0xFFFFFFFFll) && sim == (int)(g_tree_timeline_search >> 32) && half == 0;
  tree_mark<kTL>(0, tl);
  hmz_node_t* nodes = s.nodes + b * s.n_records;
  uint4* path = path_elem ? path_elem + b * (2 * kPathCap) : nullptr;
  // Before waiting for the network kernel: everything the backup needs that the PREVIOUS tree kernel wrote
  // (leaf scalars, min/max, the root's W, and the path elements = slot + entry per level, at addresses that
  // depend only on the search index: ONE round trip for paths of up to four levels).  The network kernel only
  // signals its dependents after its own wait, so that kernel has completed by the time this one runs.
  // Lane 0 of the pair owns levels 0..3 and the root, lane 1 the levels from 4 on (leaf side first).
  double mn = 0.0, mx = 0.0, root_w = 0.0;
  int pe = 0, pa = 0, depth = kPathCap + 1;
  PathBatch pb;
  pb.slot[0] = make_uint4(0u, 0u, 0u, 0u);
  bool wild = false, was_wild = false;
  const int budget = (valid && sc.budget != nullptr) ? (int)sc.budget[b] : 0x7FFFFFFF;
  const bool do_backup = !(do_select & 16) && sim < budget;  // bit 4: selection only (the first selection of a search: sim = -1)
  if (valid) {
    if (kTrusted && half == 0) was_wild = wild = wild_flags[b] != 0;
    mn = s.minmax[2 * b];
    mx = s.minmax[2 * b + 1];
  }
  if (valid && do_backup) {
    if (half == 0 && path != nullptr) load_batch4(path, 0, 4, pb);  // unconditionally: the depth is not known yet
    pe = leaf_parent[b];
    pa = leaf_action[b];
    if (path != nullptr && leaf_depth != nullptr) depth = (int)leaf_depth[b];
    if (half == 0) root_w = s.root_W[b];
    if (half == 1 && depth > 4 && depth <= kPathCap) load_batch4(path, (depth - 1) & ~3, depth, pb);
  }
  tree_mark<kTL>(1, tl, (uint32_t)(pe + pa) ^ pb.slot[0].w);
  if (kPdl) pdl_wait();  // everything below reads what the network kernel wrote
  float r_leaf = 0.f;
  double value = 0.0;
  const bool by_path = depth <= kPathCap;
  if (valid && do_backup) {
    r_leaf = ld_net_out<kPdl>(r + b);
    const float v_leaf = ld_net_out<kPdl>(v + b);
    value = (double)v_leaf;
    const float* pp = p + b * 6 + 3 * half;  // this lane's three priors
    const float q0 = ld_net_out<kPdl>(pp), q1 = ld_net_out<kPdl>(pp + 1), q2 = ld_net_out<kPdl>(pp + 2);
    write_fresh_half_vals(&nodes[sim + 1], half, q0, q1, q2, pe, pa);
    if (capture != nullptr) {  // parity tests: the network outputs this backup consumed, [p0..p5, r, v] per search
      float4* cap = reinterpret_cast<float4*>(capture + b * 8) + half;
      *cap = half == 0 ? make_float4(q0, q1, q2, ld_net_out<kPdl>(pp + 3)) : make_float4(q1, q2, r_leaf, v_leaf);
    }
    tree_mark<kTL>(6, tl, __float_as_uint(r_leaf));
    if (half == 1 && by_path && depth > 4) backup_deep(nodes, path, pb, depth, sim, r_leaf, value, discount, mn, mx, wild, tb);
  }
  {  // lane 1's running (value, min, max) to lane 0
    const int src = (threadIdx.x & 31) | 1;
    const double v1 = __shfl_sync(0xffffffffu, value, src);
    const double mn1 = __shfl_sync(0xffffffffu, mn, src);
    const double mx1 = __shfl_sync(0xffffffffu, mx, src);
    const bool wild1 = __shfl_sync(0xffffffffu, (int)wild, src) != 0;
    if (half == 0 && by_path && depth > 4) {
      value = v1;
      mn = mn1;
      mx = mx1;
      wild |= wild1;
    }
  }
  if (valid && half == 0 && do_backup) {
    tree_mark<kTL>(7, tl, (uint32_t)__double2loint(root_w) ^ (uint32_t)__double2loint(mn));
    if (by_path)
      backup_top(nodes, pb, depth, sim, r_leaf, value, discount, root_w, mn, mx, wild, tb);
    else
      backup_walk(nodes, pe, pa, sim, r_leaf, value, discount, root_w, mn, mx, wild, tb);
    if (kTrusted && wild && !was_wild) wild_flags[b] = 1;
    s.root_W[b] = root_w;
    s.minmax[2 * b] = mn;
    s.minmax[2 * b + 1] = mx;
    if (tl) {
      g_tree_timeline[2] = (unsigned long long)depth;
      tree_mark<kTL>(3, tl, (uint32_t)__double2loint(mn));
    }
  }
  if (!(do_select & 1)) return;
  // lane 0's slot stores must be visible to its partner's loads in the walk below (a shuffle orders nothing in memory)
  __syncwarp();
  // lane 0's (min, max) to its partner
  mn = __shfl_sync(0xffffffffu, mn, (threadIdx.x & 31) & ~1);
  mx = __shfl_sync(0xffffffffu, mx, (threadIdx.x & 31) & ~1);
  if (kTrusted) wild = __shfl_sync(0xffffffffu, (int)wild, (threadIdx.x & 31) & ~1) != 0;
  tree_mark<kTL>(40, tl, (uint32_t)__double2loint(mn));
  const double* rp = s.root_prior_is_f64 ? s.root_prior + b * 6 : nullptr;
  const bool sel = valid && sim + 1 < budget;  // (a search past its budget stays in the warp-uniform walk, masked)
  const Leaf leaf = select_leaf<kTL, kTrusted, TB>(nodes, rp, mn, mx, sim + 1, ucb_table, discount, half, nullptr, 0, path, tl, sel, wild, tb);
  if (half == 0 && sel) {
    leaf_parent[b] = (uint16_t)leaf.parent;
    leaf_action[b] = (uint8_t)leaf.action;
    leaf_depth[b] = (uint16_t)leaf.depth;
    // The network kernel that follows gathers the parent's latent row (written many simulations ago, long gone
    // from L2): ask for it now, a whole kernel launch ahead of its use.
    if (s.latents != nullptr) {
      const size_t row_bytes = s.latent_dtype == HMZ_LATENT_F32 ? 256 : 128;
      const char* row = reinterpret_cast<const char*>(s.latents) + ((size_t)b * s.n_records + leaf.parent) * row_bytes;
      asm volatile("prefetch.global.L2 [%0];" ::"l"(row));
      if (row_bytes == 256) asm volatile("prefetch.global.L2 [%0];" ::"l"(row + 128));
    }
    if (tl) {
      g_tree_timeline[4] = (unsigned long long)leaf.depth;
      tree_mark<kTL>(5, tl);
    }
  }
}


// MCTS/mcts.py:112-122 for one search: child_N of the root, generate_play_policy (:154-176: visits ** clamp(1/T, 1, 5)
// for T > 0, raw counts for T == 0, divided by their np.sum) and the action — np.argmax(child_visits) (first maximum,
// :117) or np.random.choice(6, p=pi) with its single uniform `u` supplied (:120: cdf / cdf[-1], searchsorted right).
// pow_table (nullable) [pow_table_len][6]: the caller's own NumPy powers of every possible count at every position of
// the 6-element visit array (see hmz_search_root_policy).
struct RootPolicy {
  int n[6];
  double prob[6];
  int action;
};
__device__ __forceinline__ RootPolicy root_policy_eval(const hmz_node_t* root, double temperature, int deterministic, double u,
                                                       const double* __restrict__ pow_table, int pow_table_len) {
  RootPolicy out;
  double w[6];
#pragma unroll
  for (int a = 0; a < 6; ++a) out.n[a] = root->h[a / 3].c[a % 3].N;
  double ex = 1.0;
  if (temperature > 0.0) ex = fmax(1.0, fmin(5.0, __ddiv_rn(1.0, temperature)));
  const int iex = (int)ex;
#pragma unroll
  for (int a = 0; a < 6; ++a) {
    const double x = (double)out.n[a];
    if (pow_table != nullptr && out.n[a] < pow_table_len) {  // visits ** exponent exactly as the caller's NumPy evaluates it
      w[a] = pow_table[out.n[a] * 6 + a];
    } else if ((double)iex == ex) {  // integer exponents 1..5: exact products while < 2^53
      double y = x;
      for (int k = 1; k < iex; ++k) y = __dmul_rn(y, x);
      w[a] = y;
    } else {
      w[a] = pow(x, ex);
    }
  }
  // np.sum of 6 doubles: left to right (NumPy sums arrays shorter than 8 sequentially; the order matters once the
  // powers pass 2^53, e.g. exponent 5 with about 1,000 visits)
  double total = w[0];
#pragma unroll
  for (int a = 1; a < 6; ++a) total = __dadd_rn(total, w[a]);
#pragma unroll
  for (int a = 0; a < 6; ++a) out.prob[a] = __ddiv_rn(w[a], total);
  int act = 0;
  if (deterministic) {
    for (int a = 1; a < 6; ++a)
      if (out.n[a] > out.n[act]) act = a;
  } else {
    double cdf[6];
    cdf[0] = out.prob[0];
#pragma unroll
    for (int a = 1; a < 6; ++a) cdf[a] = __dadd_rn(cdf[a - 1], out.prob[a]);
    const double last = cdf[5];
    act = 0;
#pragma unroll
    for (int a = 0; a < 6; ++a) act += (__ddiv_rn(cdf[a], last) <= u) ? 1 : 0;
    if (act > 5) act = 5;
  }
  out.action = act;
  return out;
}

}  // namespace hmz
