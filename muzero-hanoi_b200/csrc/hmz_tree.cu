// Tree-store kernels: pUCT selection, expansion + discounted backup, root policy (sm_100a).
//
// Restates MCTS/mcts.py:34-126 and MCTS/node.py:30-136 of the reference over the 128-byte node
// records of include/hmz.h; device-side building blocks and the arithmetic contract are in
// hmz_tree.cuh.  These kernels are latency-bound gathers (one 128-byte record per tree level, one
// 16-byte slot per backup step); there is no contraction here and nothing for tensor cores to do.
#include <cstdlib>

#include "hmz_common.cuh"
#include "hmz_net_tc.cuh"
#include "hmz_tree.cuh"

namespace hmz {

// Warps never synchronise with each other, so the block size only sets the granularity at which finished
// work frees its registers for the next block: a block lives as long as the DEEPEST of its walks.
constexpr int kTreeThreads = 128;                    // 16 searches per warp
constexpr int kSearchesPerBlock = kTreeThreads / 2;  // one lane pair per search
constexpr int kLatentWidth = HMZ_LATENT;

__global__ void __launch_bounds__(256) search_minmax_reset(double* __restrict__ minmax, int64_t n) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    minmax[2 * i] = __longlong_as_double(0x7FF0000000000000ll);      // +inf  (MCTS/utils_mcts.py:6)
    minmax[2 * i + 1] = __longlong_as_double(0xFFF0000000000000ll);  // -inf  (MCTS/utils_mcts.py:5)
  }
}

// root_node.expand(prior, h, 0.0) (MCTS/mcts.py:52-69): record 0 <- priors, everything else cleared;
// root.W <- 0.  The prior is either given (float64) or built from the network policy p0 with the
// optional Dirichlet mix of add_dirichlet_noise (MCTS/mcts.py:148-150).
__global__ void __launch_bounds__(kTreeThreads) search_begin(hmz_search_t s, const double* __restrict__ root_prior,
                                                             const float* __restrict__ p0, const double* __restrict__ noise,
                                                             float one_minus_eps, double eps) {
  const int half = threadIdx.x & 1;
  const int64_t b = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 1;
  if (b >= s.n_searches) return;
  float pr[6];
#pragma unroll
  for (int a = 0; a < 6; ++a) {
    double p;
    if (p0 != nullptr) {
      const float q = p0[b * 6 + a];
      p = (double)q;
      if (noise != nullptr)  // (1-eps)*prob is a float32 product, the sum with eps*noise is float64
        p = __dadd_rn((double)__fmul_rn(one_minus_eps, q), __dmul_rn(eps, noise[b * 6 + a]));
    } else {
      p = root_prior[b * 6 + a];
    }
    pr[a] = (float)p;
    if (half == 0 && (p0 != nullptr || s.root_prior != root_prior)) s.root_prior[b * 6 + a] = p;
  }
  write_fresh_half(&s.nodes[b * s.n_records], half, pr, 0, 0);
  if (half == 0) s.root_W[b] = 0.0;
}

// Phase 1 of one simulation for every search (one lane pair each).
__global__ void __launch_bounds__(kTreeThreads) search_select(hmz_search_t s, int sim, const double* __restrict__ ucb_table,
                                                              double discount, uint16_t* __restrict__ leaf_parent,
                                                              uint8_t* __restrict__ leaf_action,
                                                              uint16_t* __restrict__ leaf_depth, uint8_t* __restrict__ path_out,
                                                              int path_cap, uint4* __restrict__ path_elem) {
  const int half = threadIdx.x & 1;
  const int64_t b_raw = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 1;
  const bool valid = b_raw < s.n_searches;  // out-of-range pairs stay in the warp-uniform walk, masked
  const int64_t b = valid ? b_raw : s.n_searches - 1;
  const double* rp = s.root_prior_is_f64 ? s.root_prior + b * 6 : nullptr;
  const Leaf leaf = select_leaf(s.nodes + b * s.n_records, rp, s.minmax[2 * b], s.minmax[2 * b + 1], sim, ucb_table,
                                discount, half, path_out ? path_out + b * path_cap : nullptr, path_cap,
                                path_elem ? path_elem + b * (2 * kPathCap) : nullptr, false, valid);
  if (half == 0 && valid) {
    leaf_parent[b] = (uint16_t)leaf.parent;
    leaf_action[b] = (uint8_t)leaf.action;
    if (leaf_depth) leaf_depth[b] = (uint16_t)leaf.depth;
  }
}

// The fused hot-loop kernel of the launch-per-simulation schedule: tree_phase() (hmz_tree.cuh) for one lane pair per
// search, launched as a programmatic dependent of the network kernel.  Five blocks per SM: 20 warps at 96 registers.
template <bool kTL, bool kTrusted>
__global__ void __launch_bounds__(kTreeThreads, 5) search_backup_select(hmz_search_t s, int sim, const double* __restrict__ ucb_table,
                                                                     double discount, TreeScratch sc, int do_select) {
  if (threadIdx.x == 0) gantt_mark(sc.gantt, 0);
  tree_phase<kTL, kTrusted, true>(s, sim, ucb_table, discount, sc, do_select, (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 1,
                                  (int)(threadIdx.x & 1), GlobalTables());
  if ((threadIdx.x & 31) == 0) gantt_mark(sc.gantt, 1);
}

// Server schedule (HMZ_SCHEDULE_SERVER, hmz_persist.cu): the fused tree phase as an ORDINARY launch whose warps hand
// 256-search tile pairs to / from network CTAs that stay resident on their own SMs for the whole search:
//   MLP -> tree   the warps poll mlp_done[pair] until the network outputs of the simulation they back up are stored (acquire)
//   tree -> MLP   every warp adds 1 to tree_done[pair] (release) after its 16 searches' next selection
template <bool kTrusted>
__global__ void __launch_bounds__(128, 5) search_tree_served(hmz_search_t s, int sim, const double* __restrict__ ucb_table, double discount,
                                                            TreeScratch sc, int flags, uint32_t* tree_done, const uint32_t* mlp_done,
                                                            int pair_base) {
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  const int lane = threadIdx.x & 31;
  const int pair = pair_base + (int)(t >> 9);  // 512 threads = 256 searches per tile pair; a warp never straddles pairs
  if (!(flags & 16)) {  // the backup consumes the network outputs of simulation `sim`: wait for the pair's pass
    const uint32_t need = (uint32_t)sim + 1u;
    const uint32_t* flag = mlp_done + (size_t)pair * 8;
    if (lane == 0) {
      tc::WaitGuard guard;
      while (tc::v4::ld_relaxed_u32(flag) < need) {
        tc::v4::persist_backoff();
        guard.poll();
#ifdef HMZ_WATCHDOG_SOFT
        if (guard.expired) {
          if ((t & 511) == 0) printf("tree block %d: pair %d sim %d waits mlp_done >= %u, sees %u (tree_done %u)\n", (int)blockIdx.x, pair, sim, need, tc::v4::ld_relaxed_u32(flag), tc::v4::ld_relaxed_u32(tree_done + (size_t)pair * 8));
          break;
        }
#endif
      }
    }
    __syncwarp();
    tc::v4::fence_acquire_gpu();
  }
  if (threadIdx.x == 0) gantt_mark(sc.gantt, 0);
  tree_phase<false, kTrusted, false>(s, sim, ucb_table, discount, sc, flags, t >> 1, lane & 1, GlobalTables());
  if (flags & 1) {
    __syncwarp();  // every lane's stores of the slice happen before lane 0's release
    if (lane == 0) tc::v4::red_release_add(tree_done + (size_t)pair * 8, 1u);
  }
  if (lane == 0) gantt_mark(sc.gantt, 1);
}


// Node.child_Q / child_U of one node per search (inspection; same arithmetic as select_leaf).
__global__ void __launch_bounds__(128) search_child_scores(hmz_search_t s, const uint16_t* __restrict__ record,
                                                          const int32_t* __restrict__ node_n, const double* __restrict__ ucb_table,
                                                          double discount, float* __restrict__ q_out, float* __restrict__ u_out,
                                                          int32_t* __restrict__ best_out) {
  const int64_t b = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (b >= s.n_searches) return;
  const int e = record[b];
  const hmz_node_t* rec = s.nodes + b * s.n_records + e;
  const double mn = s.minmax[2 * b], mx = s.minmax[2 * b + 1];
  const bool normalise = mx > mn;
  const double range = __dsub_rn(mx, mn), tn = ucb_table[node_n[b]];
  float best_score = 0.f;
  int best = 0;
  for (int a = 0; a < 6; ++a) {
    const hmz_child_t c = rec->h[a / 3].c[a % 3];
    float qf = 0.0f;
    if (c.N > 0) {
      double q = __dadd_rn((double)c.rwd, __dmul_rn(discount, div_by_count(c.W, (int)c.N)));
      if (normalise) q = __ddiv_rn(__dsub_rn(q, mn), range);
      qf = __double2float_rn(q);
    }
    const double w = __ddiv_rn(tn, (double)(c.N + 1));
    const float u = (e == 0 && s.root_prior_is_f64) ? __double2float_rn(__dmul_rn(s.root_prior[b * 6 + a], w))
                                                    : __fmul_rn(rec->h[a / 3].prior[a % 3], __double2float_rn(w));
    q_out[b * 6 + a] = qf;
    u_out[b * 6 + a] = u;
    const float score = __fadd_rn(qf, u);
    if (a == 0 || score > best_score) {
      best_score = score;
      best = a;
    }
  }
  if (best_out) best_out[b] = best;
}

// MCTS/mcts.py:112-126 per search (one thread each; 52 bytes in, <= 76 bytes out); arithmetic in root_policy_eval().
__global__ void __launch_bounds__(256) search_root_policy(hmz_search_t s, int n_sims, double temperature,
                                                         int deterministic, const double* __restrict__ uniforms,
                                                         const double* __restrict__ pow_table, int pow_table_len,
                                                         int32_t* __restrict__ visits, double* __restrict__ pi,
                                                         double* __restrict__ root_q, int32_t* __restrict__ action,
                                                         const uint16_t* __restrict__ budget) {
  for (int64_t b = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; b < s.n_searches;
       b += (int64_t)gridDim.x * blockDim.x) {
    const RootPolicy rp = root_policy_eval(s.nodes + b * s.n_records, temperature, deterministic, deterministic ? 0.0 : uniforms[b],
                                           pow_table, pow_table_len);
    if (visits) {
#pragma unroll
      for (int a = 0; a < 6; ++a) visits[b * 6 + a] = rp.n[a];
    }
    if (pi) {
#pragma unroll
      for (int a = 0; a < 6; ++a) pi[b * 6 + a] = rp.prob[a];
    }
    const int n = budget != nullptr ? (int)budget[b] : n_sims;  // (per search in a heterogeneous batch)
    if (root_q) root_q[b] = n > 0 ? __ddiv_rn(s.root_W[b], (double)n) : 0.0;  // Node.Q (node.py:125-131)
    if (action) action[b] = rp.action;
  }
}

// Tooling / tests: the exact-division shortcuts of hmz_tree.cuh against __ddiv_rn, bit for bit, on random
// operands shaped like the search's (sums of float32-derived values over small counts, ranges of such).
__global__ void __launch_bounds__(256) div_check(uint64_t n_samples, uint64_t seed, unsigned long long* __restrict__ counters) {
  unsigned long long bad_count = 0, bad_known = 0;
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n_samples; i += (uint64_t)gridDim.x * blockDim.x) {
    const Philox4 x = philox4x32_10((uint32_t)i, (uint32_t)(i >> 32), 0x1234u, 0u, (uint32_t)seed, (uint32_t)(seed >> 32));
    const Philox4 y = philox4x32_10((uint32_t)i, (uint32_t)(i >> 32), 0x5678u, 1u, (uint32_t)seed, (uint32_t)(seed >> 32));
    // a: full random significand, exponent in [-60, 60) around 1, random sign; every 4th sample a float32 value,
    // every 16th an integer-valued double
    const unsigned long long mant = ((unsigned long long)(x.x & 0xFFFFFu) << 32) | x.y;
    const int ex = 1023 - 60 + (int)(x.z % 120u);
    double a = __longlong_as_double((long long)(((unsigned long long)(x.w & 1u) << 63) | ((unsigned long long)ex << 52) | mant));
    if ((i & 3u) == 1u) a = (double)(float)a;
    if ((i & 15u) == 2u) a = (double)(long long)(a * 1024.0);
    const int n = (i & 1u) ? 1 + (int)(y.x % 256u) : 1 + (int)(y.x % (unsigned)kRcpTable);
    if (__double_as_longlong(div_by_count(a, n)) != __double_as_longlong(__ddiv_rn(a, (double)n))) ++bad_count;
    // b: positive, exponent in [-30, 30), random significand; every 8th sample an all-ones significand
    unsigned long long bm = ((unsigned long long)(y.y & 0xFFFFFu) << 32) | y.z;
    if ((i & 7u) == 3u) bm = 0xFFFFFFFFFFFFFull;
    const double b = __longlong_as_double((long long)(((unsigned long long)(1023 - 30 + (int)(y.w % 60u)) << 52) | bm));
    const bool ok = rcp_usable(b);
    if (__double_as_longlong(div_by_known(a, b, ok ? __drcp_rn(b) : 0.0, ok)) != __double_as_longlong(__ddiv_rn(a, b))) ++bad_known;
  }
  if (bad_count) atomicAdd(&counters[0], bad_count);
  if (bad_known) atomicAdd(&counters[1], bad_known);
}

static int ensure_rcp_table();
static int ensure_tree_attrs();

int check_search(const hmz_search_t* s, const char* who) {
  if (!s) return fail(HMZ_ERR_INVALID, "%s: null search descriptor", who);
  if (s->n_searches < 0 || s->n_records < 1 || s->n_records > 65535)
    return fail(HMZ_ERR_INVALID, "%s: n_searches=%lld n_records=%d out of range", who, (long long)s->n_searches,
                s->n_records);
  if (s->n_searches > 0 && (!s->nodes || !s->root_prior || !s->root_W || !s->minmax))
    return fail(HMZ_ERR_INVALID, "%s: null buffer in search descriptor", who);
  if ((reinterpret_cast<uintptr_t>(s->nodes) & 127u) != 0)
    return fail(HMZ_ERR_INVALID, "%s: nodes must be 128-byte aligned", who);
  if (s->n_searches == 0) return HMZ_OK;
  if (int rc = ensure_tree_attrs()) return rc;
  return ensure_rcp_table();
}

// g_rcp[k] = 1.0 / k by the host's IEEE division, uploaded once per device and host thread.
static int ensure_rcp_table() {
  static thread_local int done_dev = -1;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return fail(HMZ_ERR_CUDA, "cudaGetDevice failed (no CUDA device?)");
  if (done_dev == dev) return HMZ_OK;
  static double host[kRcpTable + 1];
  host[0] = 0.0;
  for (int k = 1; k <= kRcpTable; ++k) host[k] = 1.0 / (double)k;
  static CountRow rows[kRcpTable];
  for (int n = 0; n < kRcpTable; ++n) {
    const double a = (double)(n > 0 ? n : 1), b = (double)(n + 1);
    rows[n] = CountRow{1.0 / a, 1.0 / b, a, b};
  }
  if (cudaMemcpyToSymbol(g_rcp, host, sizeof(host)) != cudaSuccess || cudaMemcpyToSymbol(g_cnt, rows, sizeof(rows)) != cudaSuccess ||
      cudaDeviceSynchronize() != cudaSuccess)
    return fail(HMZ_ERR_CUDA, "reciprocal table upload failed: %s", cudaGetErrorString(cudaGetLastError()));
  done_dev = dev;
  return HMZ_OK;
}

// The tree kernels use no shared memory, the tensor-core kernel all of it.  Left alone, the driver gives the tree
// kernels the largest L1 split and every alternation between the two kernels re-partitions the SM's L1 / shared
// memory.  Pinning the tree kernels to an explicit split removes ~1.8 us from every kernel switch (measured:
// 50.4 -> 46.7 us per simulation with serial launches; any explicit value from 0 to 75 % behaves the same, 100 %
// starves the tree kernel's L1).
constexpr int kTreeCarveoutPct = 25;  // percent of the SM's L1 / shared memory given to shared memory
static int ensure_tree_attrs() {
  static thread_local int done_dev = -1;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return fail(HMZ_ERR_CUDA, "cudaGetDevice failed (no CUDA device?)");
  if (done_dev == dev) return HMZ_OK;
  cudaError_t e = cudaFuncSetAttribute(search_backup_select<false, false>, cudaFuncAttributePreferredSharedMemoryCarveout, kTreeCarveoutPct);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(search_backup_select<false, true>, cudaFuncAttributePreferredSharedMemoryCarveout, kTreeCarveoutPct);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(search_backup_select<true, true>, cudaFuncAttributePreferredSharedMemoryCarveout, kTreeCarveoutPct);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(search_select, cudaFuncAttributePreferredSharedMemoryCarveout, kTreeCarveoutPct);
  if (e != cudaSuccess) return fail(HMZ_ERR_CUDA, "cudaFuncSetAttribute(carveout): %s", cudaGetErrorString(e));
  done_dev = dev;
  return HMZ_OK;
}

// hmz_persist.cu
int persist_read_stats(unsigned long long* host_out);
int persist_read_timeline(unsigned long long* host_out);
int64_t persist_ctl_bytes(int64_t n_searches);
bool persist_supported(const hmz_search_t* s, int mode, int n_simulations);
int persist_launch(const hmz_search_t* s, const void* weights, int n_simulations, const double* ucb_table, double discount,
                   const CountRow* cnt_table, const TreeScratch& scratch, void* ctl_mem, cudaStream_t stream);
int server_mlp_launch(const hmz_search_t* s, const void* weights, int n_simulations, TreeScratch scratch, void* ctl_mem,
                      int pairs_per_group, cudaStream_t mlp_stream, ServerCtl* out);

// Device address of this translation unit's count-row table (filled by ensure_rcp_table).
static const CountRow* count_table_address() {
  static thread_local const CountRow* addr = nullptr;
  static thread_local int addr_dev = -1;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return nullptr;
  if (addr_dev != dev) {
    void* p = nullptr;
    if (cudaGetSymbolAddress(&p, g_cnt) != cudaSuccess) return nullptr;
    addr = (const CountRow*)p;
    addr_dev = dev;
  }
  return addr;
}

static unsigned search_grid(int64_t n_searches) {
  return (unsigned)((n_searches + kSearchesPerBlock - 1) / kSearchesPerBlock);
}

// hmz_search_run's scratch in the caller's workspace (hmz_search_workspace_bytes), from its first 256-byte boundary: per
// search of the batch padded to 64 searches, p[6] r v, leaf_parent / action / depth, the sticky "wild" flag and kPathCap
// path elements of 32 B; then, at the next 256-byte boundary, the hand-off block of the persistent and server schedules
// (persist_ctl_bytes).
constexpr int64_t kScratchBytesPerSearch = 40 + 32 * kPathCap;
static int64_t padded_searches(int64_t n_searches) { return (n_searches + 63) / 64 * 64; }

struct SimScratch {
  float *p, *r, *v;
  uint16_t *lp, *depth;
  uint8_t *la, *wild;
  uint4* path;
  void* ctl;  // the hand-off block (whole batch)
};
// The scratch of a batch of n_searches, from its search `lo` on.
static SimScratch carve_scratch(void* workspace, int64_t n_searches, int64_t lo) {
  const int64_t padded_total = padded_searches(n_searches);
  char* ws = (char*)(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
  SimScratch sc;
  sc.p = (float*)ws + lo * 6;
  sc.r = (float*)(ws + padded_total * 24) + lo;
  sc.v = (float*)(ws + padded_total * 28) + lo;
  sc.lp = (uint16_t*)(ws + padded_total * 32) + lo;
  sc.la = (uint8_t*)(ws + padded_total * 34) + lo;
  sc.depth = (uint16_t*)(ws + padded_total * 36) + lo;
  sc.wild = (uint8_t*)(ws + padded_total * 38) + lo;
  sc.path = (uint4*)(ws + padded_total * 40) + lo * (2 * kPathCap);
  sc.ctl = ws + (((size_t)padded_total * kScratchBytesPerSearch + 255) & ~(size_t)255);
  return sc;
}

// The root policy of every search of `s` after n_simulations; budget (nullable, hmz_multi_t): each search's own count.
static int root_policy_launch(const hmz_search_t* s, int n_simulations, const uint16_t* budget, double temperature,
                              int deterministic, const double* uniforms, const double* pow_table, int32_t* visits, double* pi,
                              double* root_q, int32_t* action, void* stream) {
  search_root_policy<<<grid_for(s->n_searches, 256, 4), 256, 0, (cudaStream_t)stream>>>(
      *s, n_simulations, temperature, deterministic, uniforms, pow_table, n_simulations + 1, visits, pi, root_q, action, budget);
  return check_launch("search_root_policy");
}

}  // namespace hmz

using namespace hmz;

static long long g_tree_tl_search = -1;  // host copy of g_tree_timeline_search (tooling)

extern "C" {

// Tooling only: search >= 0 makes hmz_search_run launch the instrumented instantiation of the fused
// backup + select kernel, whose lane pair `search` records clock64() at its phase boundaries; host_out
// (nullable) receives the 64 marks of the last launch.
int hmz_debug_div_check(uint64_t n_samples, uint64_t seed, unsigned long long* counters, void* stream) {
  if (!counters) return fail(HMZ_ERR_INVALID, "hmz_debug_div_check: null counters");
  if (int rc = ensure_rcp_table()) return rc;
  div_check<<<grid_for((int64_t)n_samples, 256 * 64, 8), 256, 0, (cudaStream_t)stream>>>(n_samples, seed, counters);
  return check_launch("div_check");
}

int hmz_debug_persist_timeline(unsigned long long* host_out) {
  if (!host_out) return fail(HMZ_ERR_INVALID, "hmz_debug_persist_timeline: null pointer");
  return persist_read_timeline(host_out);
}

int hmz_debug_persist_stats(unsigned long long* host_out) {
  if (!host_out) return fail(HMZ_ERR_INVALID, "hmz_debug_persist_stats: null pointer");
  return persist_read_stats(host_out);
}

int hmz_debug_tree_timeline(long long search, unsigned long long* host_out) {
  if (host_out && cudaMemcpyFromSymbol(host_out, g_tree_timeline, sizeof(unsigned long long) * 64) != cudaSuccess)
    return fail(HMZ_ERR_CUDA, "hmz_debug_tree_timeline: cudaMemcpyFromSymbol failed");
  if (cudaMemcpyToSymbol(g_tree_timeline_search, &search, sizeof(search)) != cudaSuccess)
    return fail(HMZ_ERR_CUDA, "hmz_debug_tree_timeline: cudaMemcpyToSymbol failed");
  g_tree_tl_search = search;
  return HMZ_OK;
}

// Non-default compile-time switches of this build ("" for a clean build), so that tests and bench lines can tell a
// tooling or A/B build from the shipped one.  None of them changes results.
const char* hmz_build_flags(void) {
  return ""
#ifdef HMZ_PERSIST_STATS
         " HMZ_PERSIST_STATS"
#endif
#ifdef HMZ_VARIANT
         " HMZ_VARIANT"
#endif
      ;
}

int64_t hmz_search_workspace_bytes(int64_t n_searches) {
  if (n_searches < 0) return -1;
  // carve_scratch's layout; 1024 covers the two 256-byte alignments
  return padded_searches(n_searches) * kScratchBytesPerSearch + 1024 + persist_ctl_bytes(n_searches);
}

int hmz_search_minmax_reset(double* minmax, int64_t n, void* stream) {
  ProfScope prof_scope(HMZ_PROF_OTHER, stream);
  if (n == 0) return HMZ_OK;
  if (!minmax || n < 0) return fail(HMZ_ERR_INVALID, "hmz_search_minmax_reset: bad arguments");
  search_minmax_reset<<<grid_for(n, 256, 8), 256, 0, (cudaStream_t)stream>>>(minmax, n);
  return check_launch("search_minmax_reset");
}

int hmz_search_begin(const hmz_search_t* s, const double* root_prior, void* stream) {
  ProfScope prof_scope(HMZ_PROF_OTHER, stream);
  if (int rc = check_search(s, "hmz_search_begin")) return rc;
  if (s->n_searches == 0) return HMZ_OK;
  if (!root_prior) return fail(HMZ_ERR_INVALID, "hmz_search_begin: null root_prior");
  search_begin<<<search_grid(s->n_searches), kTreeThreads, 0, (cudaStream_t)stream>>>(*s, root_prior, nullptr, nullptr, 0.f, 0.0);
  return check_launch("search_begin");
}

int hmz_search_begin_p0(const hmz_search_t* s, const float* p0, const double* noise, double eps, void* stream) {
  ProfScope prof_scope(HMZ_PROF_OTHER, stream);
  if (int rc = check_search(s, "hmz_search_begin_p0")) return rc;
  if (s->n_searches == 0) return HMZ_OK;
  if (!p0) return fail(HMZ_ERR_INVALID, "hmz_search_begin_p0: null p0");
  if ((noise != nullptr) != (s->root_prior_is_f64 != 0))
    return fail(HMZ_ERR_INVALID, "hmz_search_begin_p0: root_prior_is_f64 must be set iff noise is given");
  search_begin<<<search_grid(s->n_searches), kTreeThreads, 0, (cudaStream_t)stream>>>(*s, nullptr, p0, noise,
                                                                                   (float)(1.0 - eps), eps);
  return check_launch("search_begin_p0");
}

int hmz_search_select(const hmz_search_t* s, int sim, const double* ucb_table, double discount, uint16_t* leaf_parent,
                      uint8_t* leaf_action, uint16_t* leaf_depth, uint8_t* path_out, int path_cap, void* stream) {
  ProfScope prof_scope(HMZ_PROF_SELECT, stream);
  if (int rc = check_search(s, "hmz_search_select")) return rc;
  if (s->n_searches == 0) return HMZ_OK;
  if (!ucb_table || !leaf_parent || !leaf_action || sim < 0 || sim + 1 >= s->n_records || (path_out && path_cap < 1))
    return fail(HMZ_ERR_INVALID, "hmz_search_select: bad arguments (sim=%d, n_records=%d)", sim, s->n_records);
  search_select<<<search_grid(s->n_searches), kTreeThreads, 0, (cudaStream_t)stream>>>(
      *s, sim, ucb_table, discount, leaf_parent, leaf_action, leaf_depth, path_out, path_cap, nullptr);
  return check_launch("search_select");
}

int hmz_search_child_scores(const hmz_search_t* s, const uint16_t* record, const int32_t* node_n, const double* ucb_table,
                            double discount, float* q_out, float* u_out, int32_t* best_out, void* stream) {
  ProfScope prof_scope(HMZ_PROF_OTHER, stream);
  if (int rc = check_search(s, "hmz_search_child_scores")) return rc;
  if (s->n_searches == 0) return HMZ_OK;
  if (!record || !node_n || !ucb_table || !q_out || !u_out)
    return fail(HMZ_ERR_INVALID, "hmz_search_child_scores: null pointer");
  search_child_scores<<<(unsigned)((s->n_searches + 127) / 128), 128, 0, (cudaStream_t)stream>>>(
      *s, record, node_n, ucb_table, discount, q_out, u_out, best_out);
  return check_launch("search_child_scores");
}

int hmz_search_expand_backup(const hmz_search_t* s, int sim, double discount, const uint16_t* leaf_parent,
                             const uint8_t* leaf_action, const float* r, const float* p, const float* v,
                             void* stream) {
  ProfScope prof_scope(HMZ_PROF_EXPAND_BACKUP, stream);
  if (int rc = check_search(s, "hmz_search_expand_backup")) return rc;
  if (s->n_searches == 0) return HMZ_OK;
  if (!leaf_parent || !leaf_action || !r || !p || !v || sim < 0 || sim + 1 >= s->n_records)
    return fail(HMZ_ERR_INVALID, "hmz_search_expand_backup: bad arguments (sim=%d, n_records=%d)", sim, s->n_records);
  // split-phase form: no recorded path, the backup walks the parent links
  TreeScratch sc{const_cast<uint16_t*>(leaf_parent), const_cast<uint8_t*>(leaf_action), nullptr, nullptr, nullptr, r, p, v, nullptr, nullptr};
  search_backup_select<false, false><<<search_grid(s->n_searches), kTreeThreads, 0, (cudaStream_t)stream>>>(*s, sim, nullptr, discount, sc, 0);
  return check_launch("search_expand_backup");
}

int hmz_search_root_policy(const hmz_search_t* s, int n_simulations, double temperature, int deterministic,
                           const double* uniforms, const double* pow_table, int32_t* visits, double* pi, double* root_q,
                           int32_t* action, void* stream) {
  ProfScope prof_scope(HMZ_PROF_ROOT_POLICY, stream);
  if (int rc = check_search(s, "hmz_search_root_policy")) return rc;
  if (!(temperature >= 0.0 && temperature <= 1.0))  // MCTS/mcts.py:163-166 -> ValueError in the Python shim
    return fail(HMZ_ERR_INVALID, "Expect `temperature` to be in the range [0.0, 1.0], got %g", temperature);
  if (s->n_searches == 0) return HMZ_OK;
  if (!deterministic && !uniforms) return fail(HMZ_ERR_INVALID, "hmz_search_root_policy: sampling needs uniforms");
  return root_policy_launch(s, n_simulations, nullptr, temperature, deterministic, uniforms, pow_table, visits, pi, root_q,
                            action, stream);
}

int hmz_search_root_policy_multi(const hmz_search_t* s, const hmz_multi_t* m, double temperature, int deterministic,
                                 const double* uniforms, const double* pow_table, int32_t* visits, double* pi, double* root_q,
                                 int32_t* action, void* stream) {
  ProfScope prof_scope(HMZ_PROF_ROOT_POLICY, stream);
  if (!s) return fail(HMZ_ERR_INVALID, "hmz_search_root_policy_multi: null search descriptor");
  if (int rc = check_multi(m, s->n_searches, -1, s->n_records, true, "hmz_search_root_policy_multi")) return rc;
  if (!(temperature >= 0.0 && temperature <= 1.0))
    return fail(HMZ_ERR_INVALID, "Expect `temperature` to be in the range [0.0, 1.0], got %g", temperature);
  if (s->n_searches == 0) return HMZ_OK;
  if (!deterministic && !uniforms) return fail(HMZ_ERR_INVALID, "hmz_search_root_policy_multi: sampling needs uniforms");
  if (int rc = check_search(s, "hmz_search_root_policy_multi")) return rc;
  return root_policy_launch(s, m->host_block_budget[0], m->budget, temperature, deterministic, uniforms, pow_table, visits, pi,
                            root_q, action, stream);
}

namespace {
struct GroupStreams {
  int dev = -1;
  cudaStream_t stream[16] = {};
  cudaEvent_t done[16] = {};
  cudaEvent_t fork = nullptr;
  int n = 0;
};
// Lazily created, per host thread and device; lives for the life of the process.
int get_group_streams(int want, GroupStreams** out) {
  static thread_local GroupStreams gs;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return fail(HMZ_ERR_CUDA, "cudaGetDevice failed");
  if (gs.dev != dev) {
    gs = GroupStreams();
    gs.dev = dev;
  }
  if (!gs.fork && cudaEventCreateWithFlags(&gs.fork, cudaEventDisableTiming) != cudaSuccess)
    return fail(HMZ_ERR_CUDA, "cudaEventCreate failed");
  while (gs.n < want) {
    if (cudaStreamCreateWithFlags(&gs.stream[gs.n], cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&gs.done[gs.n], cudaEventDisableTiming) != cudaSuccess)
      return fail(HMZ_ERR_CUDA, "cudaStreamCreate failed");
    ++gs.n;
  }
  *out = &gs;
  return HMZ_OK;
}

// Helper streams forked from the caller's stream: begin(n) orders n of them behind the work enqueued on it so far, and the
// destructor joins every forked one back into it — on every path, errors included, so that the caller's stream stays
// ordered behind whatever was enqueued on them.
class StreamFork {
 public:
  explicit StreamFork(cudaStream_t caller) : caller_(caller) {}
  int begin(int n) {
    if (int rc = get_group_streams(n, &gs_)) return rc;
    if (cudaEventRecord(gs_->fork, caller_) != cudaSuccess) return fail(HMZ_ERR_CUDA, "cudaEventRecord(fork) failed");
    for (; forked_ < n; ++forked_)
      if (cudaStreamWaitEvent(gs_->stream[forked_], gs_->fork, 0) != cudaSuccess) return fail(HMZ_ERR_CUDA, "cudaStreamWaitEvent failed");
    return HMZ_OK;
  }
  cudaStream_t operator[](int g) const { return gs_->stream[g]; }
  ~StreamFork() {
    for (int g = 0; g < forked_; ++g) {
      cudaEventRecord(gs_->done[g], gs_->stream[g]);
      cudaStreamWaitEvent(caller_, gs_->done[g], 0);
    }
  }

 private:
  cudaStream_t caller_;
  GroupStreams* gs_ = nullptr;
  int forked_ = 0;
};

// Searches [lo, hi) of `s` as a descriptor of their own (their scratch: carve_scratch(s->workspace, s->n_searches, lo)).
hmz_search_t search_slice(const hmz_search_t* s, int64_t lo, int64_t hi) {
  const size_t lat_elem = s->latent_dtype == HMZ_LATENT_F32 ? 4 : 2;
  hmz_search_t sub = *s;
  sub.nodes = s->nodes + lo * s->n_records;
  sub.latents = (char*)s->latents + (size_t)lo * s->n_records * kLatentWidth * lat_elem;
  sub.root_prior = s->root_prior + lo * 6;
  sub.root_W = s->root_W + lo;
  sub.minmax = s->minmax + 2 * lo;
  sub.n_searches = hi - lo;
  return sub;
}
}  // namespace


// One tree launch of the server schedule for the searches of `s` (a slice that starts at tile pair `pair_base`):
// item `sim_item` = expansion + backup of simulation sim_item - 1 (none for 0) and the selection of simulation sim_item
// (none after the last one).
static int server_tree_launch(const hmz_search_t* s, int sim_item, int n_simulations, const double* ucb_table, double discount,
                       const TreeScratch& sc, const ServerCtl& ctl, int pair_base, cudaStream_t stream) {
  const int64_t pairs = (s->n_searches + 2 * tc::kM - 1) / (2 * tc::kM);
  const int flags = (sim_item < n_simulations ? 1 : 0) | (sim_item == 0 ? 16 : 0);
  search_tree_served<true><<<dim3((unsigned)(pairs * 4)), dim3(128), 0, stream>>>(*s, sim_item - 1, ucb_table, discount, sc, flags,
                                                                               ctl.tree_done, ctl.mlp_done, pair_base);
  return check_launch("search_tree_served");
}

static int debug_skip() {
  const char* e = getenv("HMZ_DEBUG_SKIP");
  return e ? atoi(e) : 0;
}

// Weight sets and budgets of one group's searches in a heterogeneous batch (hmz_search_run_multi); all null otherwise.
struct GroupSets {
  const uint16_t* block_set;  // of the group's first block
  int64_t weight_stride;
  const uint16_t* budget;     // of the group's first search
};

// One simulation of one group: [select (first simulation only)] -> g+f MLP -> fused backup + next select.
// capture_stride / capture_lo: searches per capture row (the whole batch) and this group's first search in it.
static int run_one_sim(const hmz_search_t* s, const SimScratch& sc, const void* weights, int mode, int sim,
                       int n_simulations, const double* ucb_table, double discount, void* stream, int64_t capture_stride,
                       int64_t capture_lo, const GroupSets& sets, bool allow_head_split) {
  const int64_t B = s->n_searches;
  cudaStream_t st = (cudaStream_t)stream;
  if (sim == 0) {
    ProfScope prof_scope(HMZ_PROF_SELECT, stream);
    if (cudaMemsetAsync(sc.wild, 0, (size_t)B, st) != cudaSuccess) return fail(HMZ_ERR_CUDA, "cudaMemsetAsync(wild flags) failed");
    search_select<<<search_grid(B), kTreeThreads, 0, st>>>(*s, 0, ucb_table, discount, sc.lp, sc.la, sc.depth, nullptr, 0,
                                                          sc.path);
    if (int rc = check_launch("search_select")) return rc;
  }
  // tooling (tools/persist_probe.py): HMZ_DEBUG_SKIP=1 leaves out the network launches, =2 the tree launches — timing of
  // one kernel family alone under the group schedule; the search results are meaningless then
  const int skip = debug_skip();
  if (!(skip & 1)) {
    ProfScope prof_scope(HMZ_PROF_NET_RECURRENT, stream);
    if (int rc = net_recurrent_sets(weights, sets.block_set, sets.weight_stride, allow_head_split, mode, s->latents, s->n_records,
                                    sc.lp, sc.la, s->latents, s->n_records, sim + 1, s->latent_dtype, sc.r, sc.p, sc.v, B, stream))
      return rc;
  }
  if (skip & 2) return HMZ_OK;
  ProfScope prof_scope(HMZ_PROF_EXPAND_BACKUP, stream);
  const int do_select = sim + 1 < n_simulations ? 1 : 0;
  const float *cr = sc.r, *cp = sc.p, *cv = sc.v;
  TreeScratch ts{sc.lp, sc.la, sc.depth, sc.path, sc.wild, cr, cp, cv,
                 s->capture ? s->capture + ((size_t)sim * (size_t)capture_stride + (size_t)capture_lo) * 8 : nullptr,
                 gantt_next(1, gantt_context_tag()), sets.budget};
  cudaError_t e = launch_pdl(g_tree_tl_search >= 0 ? search_backup_select<true, true> : search_backup_select<false, true>,
                             dim3(search_grid(B)), dim3(kTreeThreads), 0, st, *s, sim, ucb_table, discount, ts, do_select);
  if (e != cudaSuccess) return fail(HMZ_ERR_CUDA, "search_backup_select launch: %s", cudaGetErrorString(e));
  return check_launch("search_backup_select");
}

// HMZ_SCHEDULE_SERVER | k: resident network CTAs + one ordinary tree launch per simulation and stream group (k groups of
// whole tile pairs; 0 = 4).  Stream plan: the control block is zeroed on the caller's stream; the MLP stream and the k
// tree streams fork from it; the caller's stream joins all of them.
static int search_run_server(const hmz_search_t* s, const void* weights, int n_simulations, const double* ucb_table,
                             double discount, void* stream) {
  const int64_t B = s->n_searches;
  int groups = s->schedule - HMZ_SCHEDULE_SERVER;
  if (groups < 0 || groups > 15) return fail(HMZ_ERR_INVALID, "hmz_search_run: bad server schedule %d", s->schedule);
  if (groups == 0) groups = 4;
  const int64_t per = ((B + groups - 1) / groups + 255) / 256 * 256;  // whole tile pairs: the hand-offs are per pair
  groups = (int)((B + per - 1) / per);
  cudaStream_t main_stream = (cudaStream_t)stream;
  const SimScratch sc0 = carve_scratch(s->workspace, B, 0);
  if (cudaMemsetAsync(sc0.wild, 0, (size_t)B, main_stream) != cudaSuccess ||
      cudaMemsetAsync(sc0.ctl, 0, (size_t)persist_ctl_bytes(B), main_stream) != cudaSuccess)
    return fail(HMZ_ERR_CUDA, "cudaMemsetAsync(server control block) failed");
  StreamFork fork(main_stream);  // streams [0, groups): tree launches; stream `groups`: the MLP CTAs
  if (int rc = fork.begin(groups + 1)) return rc;
  {  // CUDA loads kernels lazily, and loading one may wait for the device to go idle — which the resident network CTAs
     // never let it: the tree kernel must be loaded BEFORE they are launched
    static thread_local int loaded_dev = -1;
    int dev = 0;
    cudaFuncAttributes fa;
    if (cudaGetDevice(&dev) != cudaSuccess || (loaded_dev != dev && cudaFuncGetAttributes(&fa, search_tree_served<true>) != cudaSuccess))
      return fail(HMZ_ERR_CUDA, "hmz_search_run: loading the served tree kernel failed");
    loaded_dev = dev;
  }
  ServerCtl sctl{};
  TreeScratch whole{sc0.lp, sc0.la, sc0.depth, sc0.path, sc0.wild, sc0.r, sc0.p, sc0.v, nullptr, nullptr};
  int rc = server_mlp_launch(s, weights, n_simulations, whole, sc0.ctl, (int)(per / 256), fork[groups], &sctl);
  // A tree launch that is resident before its pairs' network outputs exist holds its SM slots spinning: the group's
  // stream waits (cuStreamWaitValue32, resolved through the runtime so that libcuda is not a link dependency) until the
  // network CTAs have finished every pair of the group for the previous simulation.  Without that entry point the tree
  // warps only spin.
  typedef int (*WaitValue32)(cudaStream_t, unsigned long long, unsigned int, unsigned int);
  static WaitValue32 wait_value = nullptr;
  static bool resolved = false;
  if (!resolved) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qr;
    if (cudaGetDriverEntryPoint("cuStreamWaitValue32", &fn, cudaEnableDefault, &qr) == cudaSuccess && qr == cudaDriverEntryPointSuccess)
      wait_value = (WaitValue32)fn;
    else
      cudaGetLastError();
    resolved = true;
  }
  hmz_search_t sub[16];
  SimScratch sc[16];
  for (int g = 0; g < groups; ++g) {
    const int64_t lo = g * per;
    sub[g] = search_slice(s, lo, lo + per < B ? lo + per : B);
    sc[g] = carve_scratch(s->workspace, B, lo);
  }
  // item k: expansion + backup of simulation k - 1 (none for k = 0) and the selection of simulation k (none for k = S)
  for (int k = 0; k <= n_simulations && rc == HMZ_OK; ++k)
    for (int g = 0; g < groups && rc == HMZ_OK; ++g) {
      ProfScope prof_scope(HMZ_PROF_EXPAND_BACKUP, (void*)fork[g]);
      gantt_set_context(g, k);
      TreeScratch ts{sc[g].lp, sc[g].la, sc[g].depth, sc[g].path, sc[g].wild, sc[g].r, sc[g].p, sc[g].v,
                     (s->capture && k > 0) ? s->capture + ((size_t)(k - 1) * (size_t)B + (size_t)(g * per)) * 8 : nullptr,
                     gantt_next(1, gantt_context_tag())};
      if (wait_value && k > 0) {
        const unsigned int pairs_g = (unsigned int)((sub[g].n_searches + 255) / 256);
        if (wait_value(fork[g], (unsigned long long)(uintptr_t)(sctl.group_done + (size_t)g * 8), pairs_g * (unsigned int)k, 0u /* >= */) != 0)
          rc = fail(HMZ_ERR_CUDA, "cuStreamWaitValue32 failed");
      }
      if (rc == HMZ_OK)
        rc = server_tree_launch(&sub[g], k, n_simulations, ucb_table, discount, ts, sctl, (int)(g * per / 256), fork[g]);
    }
  return rc;
}

// The stream-group schedules (0, 1..16) of hmz_search_run and hmz_search_run_multi.  Searches never interact, so the
// batch is cut into groups whose select -> MLP -> backup chains run on separate streams: the latency-bound tree kernels of
// one group fill the issue slots the tensor-core kernel of another leaves idle.  One group runs on the caller's stream.
//   m == nullptr   group boundaries are multiples of 128 searches; every simulation runs over the whole batch.
//   m (hmz_multi_t) group boundaries are whole 256-search blocks (a block's weight set is per tile pair), each group carries
//                  its weight sets and budgets, and simulation `sim` launches over the active prefix only — the blocks
//                  whose budget exceeds sim; a group whose slice has left the prefix issues nothing, so in the late
//                  simulations fewer groups overlap.
static int search_run_groups(const hmz_search_t* s, const hmz_multi_t* m, const void* weights, int mode, int n_simulations,
                             const double* ucb_table, double discount, void* stream) {
  const int64_t B = s->n_searches;
  int groups = s->schedule;
  // measured on the B200 (tools/gpu_round.sh groupsweep, S = 100): 8,192 searches 2.08 / 2.12 / 2.17 ms per move with 1 / 2 / 4
  // groups, 16,384: 2.26 / 2.25 / 2.29, 32,768: 2.53 / 2.52 / 2.58, 65,536: 4.70 / 4.15 / 4.10 (3 groups 4.07, 6: 4.12, 8: 4.17)
  if (groups == 0) groups = B >= 49152 ? 4 : (B >= 12288 ? 2 : 1);
  const int64_t unit = m ? 256 : 128;
  const int64_t per = ((B + groups - 1) / groups + unit - 1) / unit * unit;
  groups = (int)((B + per - 1) / per);
  StreamFork fork((cudaStream_t)stream);
  if (groups > 1)
    if (int rc = fork.begin(groups)) return rc;
  hmz_search_t sub[16];
  SimScratch sc[16];
  GroupSets sets[16] = {};
  for (int g = 0; g < groups; ++g) {
    const int64_t lo = g * per;
    sub[g] = search_slice(s, lo, lo + per < B ? lo + per : B);
    sc[g] = carve_scratch(s->workspace, B, lo);
    if (m) sets[g] = GroupSets{m->block_set + lo / 256, m->weight_stride, m->budget + lo};
  }
  int64_t active = B, active_blocks = B / 256;
  int rc = HMZ_OK;
  for (int sim = 0; sim < n_simulations && rc == HMZ_OK; ++sim) {
    if (m) {
      while (active_blocks > 0 && m->host_block_budget[active_blocks - 1] <= sim) --active_blocks;
      active = active_blocks * 256;
    }
    for (int g = 0; g < groups && g * per < active && rc == HMZ_OK; ++g) {
      hmz_search_t part = sub[g];
      if (part.n_searches > active - g * per) part.n_searches = active - g * per;
      gantt_set_context(g, sim);
      // several groups in flight: the other groups' launches want the idle SMs — no head split then
      rc = run_one_sim(&part, sc[g], weights, mode, sim, n_simulations, ucb_table, discount, groups > 1 ? (void*)fork[g] : stream,
                       B, g * per, sets[g], groups == 1);
    }
  }
  return rc;
}

int hmz_search_run(const hmz_search_t* s, const void* weights, int mode, int n_simulations, const double* ucb_table,
                   double discount, void* stream) {
  if (int rc = check_search(s, "hmz_search_run")) return rc;
  if (s->n_searches == 0 || n_simulations == 0) return HMZ_OK;
  if (!weights || !ucb_table || !s->workspace || !s->latents || n_simulations < 0 ||
      n_simulations + 1 > s->n_records)
    return fail(HMZ_ERR_INVALID, "hmz_search_run: bad arguments (n_simulations=%d, n_records=%d)", n_simulations,
                s->n_records);
  const bool can_persist = persist_supported(s, mode, n_simulations);
  if (s->schedule == HMZ_SCHEDULE_PERSISTENT) {  // ONE persistent role-specialised kernel for the whole search (hmz_persist.cu)
    if (!can_persist)
      return fail(HMZ_ERR_UNSUPPORTED, "hmz_search_run: the persistent schedule needs HMZ_MODE_BF16 and n_simulations <= 2046");
    ProfScope prof_scope(HMZ_PROF_SEARCH_PERSISTENT, stream);
    const SimScratch sc = carve_scratch(s->workspace, s->n_searches, 0);
    if (cudaMemsetAsync(sc.wild, 0, (size_t)s->n_searches, (cudaStream_t)stream) != cudaSuccess) return fail(HMZ_ERR_CUDA, "cudaMemsetAsync(wild flags) failed");
    const CountRow* cnt = count_table_address();
    if (!cnt) return fail(HMZ_ERR_CUDA, "cudaGetSymbolAddress(count table) failed");
    TreeScratch ts{sc.lp, sc.la, sc.depth, sc.path, sc.wild, sc.r, sc.p, sc.v, nullptr, nullptr};
    return persist_launch(s, weights, n_simulations, ucb_table, discount, cnt, ts, sc.ctl, (cudaStream_t)stream);
  }
  if (s->schedule >= HMZ_SCHEDULE_SERVER) {
    if (!can_persist) return fail(HMZ_ERR_UNSUPPORTED, "hmz_search_run: the server schedule needs HMZ_MODE_BF16 and n_simulations <= 2046");
    return search_run_server(s, weights, n_simulations, ucb_table, discount, stream);
  }
  if (s->schedule < 0 || s->schedule > 16)
    return fail(HMZ_ERR_INVALID, "hmz_search_run: schedule %d is neither a group count in [0, 16] nor HMZ_SCHEDULE_PERSISTENT", s->schedule);
  return search_run_groups(s, nullptr, weights, mode, n_simulations, ucb_table, discount, stream);
}

int hmz_search_run_multi(const hmz_search_t* s, const hmz_multi_t* m, const void* weights, int mode, const double* ucb_table,
                         double discount, void* stream) {
  // argument errors first, before check_search makes its first CUDA call
  if (!s) return fail(HMZ_ERR_INVALID, "hmz_search_run_multi: null search descriptor");
  if (int rc = check_multi(m, s->n_searches, mode, s->n_records, true, "hmz_search_run_multi")) return rc;
  if (s->schedule == HMZ_SCHEDULE_PERSISTENT || s->schedule >= HMZ_SCHEDULE_SERVER)
    return fail(HMZ_ERR_UNSUPPORTED, "hmz_search_run_multi: only the stream-group schedules (0, 1..16) serve heterogeneous batches");
  if (s->schedule < 0 || s->schedule > 16)
    return fail(HMZ_ERR_INVALID, "hmz_search_run_multi: schedule %d is not a group count in [0, 16]", s->schedule);
  if (s->n_searches > 0 && (!weights || !ucb_table || !s->workspace || !s->latents))
    return fail(HMZ_ERR_INVALID, "hmz_search_run_multi: null argument");
  if (int rc = check_search(s, "hmz_search_run_multi")) return rc;
  if (s->n_searches == 0) return HMZ_OK;
  return search_run_groups(s, m, weights, mode, m->host_block_budget[0], ucb_table, discount, stream);
}

}  // extern "C"
