// The persistent, role-specialised search kernel (hmz_search_t.schedule = HMZ_SCHEDULE_PERSISTENT): ONE launch runs
// every simulation of MCTS.run_mcts (MCTS/mcts.py:71-109) for the whole batch, instead of two launches per simulation
// and stream group.
//
//   CTAs [0, n_mlp)         MLP role: net_tc_body<recurrent, persistent> (hmz_net_tc.cuh) — the tcgen05 g + f kernel body;
//                           CTA c owns the 256-search tile pairs c, c + n_mlp, ... and runs them once per simulation.
//   CTAs [n_mlp, gridDim)   tree role: 24 independent warps; a warp takes a TICKET (one atomic add), waits for the work item
//                           the ticket names — (tile pair, simulation), 16 tickets of 16 searches each per item — and runs
//                           tree_phase() (hmz_tree.cuh): expansion + backup of simulation s - 1 and the selection of
//                           simulation s, exactly the code of the stand-alone fused kernel.
//
// Hand-off (PersistCtl, global memory, zeroed before the launch):
//   tree -> MLP   every warp that finishes a slice adds 1 to tree_done[pair] with a GPU-scope release; the pair's MLP
//                 pass for simulation s starts when the counter reaches 16 (s + 1) (acquire).
//   MLP -> tree   when every output of the pass (r, p, v, latent rows) has been stored, one thread publishes the item
//                 (pair, s + 1) into a ticket-ordered queue with a release store; the 16 warps holding its tickets acquire it.
// Dependencies are therefore per 256 searches instead of per launch: no launch gaps, no partial last wave of tree blocks,
// no prologue / tail of the tensor-core kernel per simulation, and both roles stay busy on their own SMs for the whole move.
//
// All CTAs must be co-resident (they wait on one another): the kernel is launched cooperatively with one CTA per SM.
// Every wait on global memory is bounded; a wait that exceeds the bound traps (the launch fails) instead of hanging the GPU.
#include <cstdlib>

#include "hmz_net_tc.cuh"
#include "hmz_tree.cuh"

namespace hmz {

#ifndef HMZ_PERSIST_THREADS
#define HMZ_PERSIST_THREADS 768
#endif
constexpr int kPersistThreads = HMZ_PERSIST_THREADS;  // 24 warps; at this block size ptxas may use 80 registers per thread
constexpr int kPersistWarps = kPersistThreads / 32;

struct PersistArgs {
  hmz_search_t s;
  tc::v4::TcArgs net;
  tc::v4::PersistCtl ctl;
  const CountRow* cnt_table;  // the global count-row table (hmz_tree.cu's copy), staged into shared memory by the tree CTAs
  const double* ucb_table;
  double discount;
  TreeScratch sc;             // capture = row of simulation 0
  int64_t capture_stride;     // floats between two simulations' capture rows (0 when capture is off)
  uint32_t total_tickets;     // 16 * n_pairs * (n_sims + 1)
  int n_mlp, n_sims, n_pairs, table_rows;
};

// Tooling (HMZ_PERSIST_STATS=1): clock64 sums of the last launch — [0] tree warps waiting for an item, [1] tree warps
// working, [2] items x slices processed, [3] tree warp lifetimes, [4] MLP CTAs waiting for the tree (one thread per CTA),
// [5] MLP CTAs first push -> last push, [6] MLP passes, [7] CTAs x warps of the tree role.
static __device__ unsigned long long g_persist_stats[16];

__device__ __forceinline__ void tree_role(const PersistArgs& a, uint8_t* smem_raw) {
  // constant tables -> shared memory (the acquire at every hand-off invalidates L1)
  CountRow* s_cnt = reinterpret_cast<CountRow*>((reinterpret_cast<uintptr_t>(smem_raw) + 127) & ~(uintptr_t)127);
  double* s_ucb = reinterpret_cast<double*>(s_cnt + a.table_rows);
  for (int i = threadIdx.x; i < a.table_rows * 4; i += blockDim.x)
    reinterpret_cast<double*>(s_cnt)[i] = reinterpret_cast<const double*>(a.cnt_table)[i];
  for (int i = threadIdx.x; i < a.table_rows; i += blockDim.x) s_ucb[i] = a.ucb_table[i];
  __syncthreads();
#ifdef HMZ_PERSIST_GLOBAL_TABLES  // A/B switch: read the tables from global memory through L1 instead
  const SmemTables tb{a.cnt_table, a.ucb_table, a.table_rows};
#else
  const SmemTables tb{s_cnt, s_ucb, a.table_rows};
#endif
  const int lane = threadIdx.x & 31, half = lane & 1;
  const tc::v4::PersistCtl& pc = a.ctl;
  const bool stats = tc::v4::kPersistStats && pc.stats != nullptr && lane == 0;
  long long t_wait = 0, t_work = 0, n_items = 0;
  const long long t_begin = stats ? clock64() : 0;
  for (;;) {
    const long long c0 = stats ? clock64() : 0;
    uint32_t ticket = 0;
    if (lane == 0) ticket = atomicAdd(pc.tree_head, 1u);
    ticket = __shfl_sync(0xffffffffu, ticket, 0);
    if (ticket >= a.total_tickets) break;
    ++n_items;
    const uint32_t item = ticket / tc::v4::kSlicesPerPair, slice = ticket % tc::v4::kSlicesPerPair;
    int pair, sim;
    if (item < (uint32_t)a.n_pairs) {  // implicit items: the first selection of every pair
      pair = (int)item;
      sim = 0;
    } else {
      const unsigned long long* slot = pc.queue + ((item - (uint32_t)a.n_pairs) & pc.q_mask);
      unsigned long long q;
      tc::WaitGuard guard;
      while ((uint32_t)((q = tc::v4::ld_relaxed_u64(slot)) >> 32) != item + 1u) {
        tc::v4::persist_backoff();
        guard.poll();
      }
      pair = (int)(q & 0xFFFFu);
      sim = (int)((q >> 16) & 0xFFFFu);
    }
    tc::v4::fence_acquire_gpu();  // every lane: the item's network outputs, and whatever other SMs wrote to this slice's tree
    const long long c1 = stats ? clock64() : 0;
    const int64_t b_raw = (int64_t)pair * (2 * tc::kM) + (int64_t)slice * 16 + (lane >> 1);
    TreeScratch sc = a.sc;
    if (sc.capture != nullptr && sim > 0) sc.capture += (size_t)(sim - 1) * (size_t)a.capture_stride;
    // item (pair, sim): expansion + backup of simulation sim - 1 (none for sim = 0), selection of simulation sim (none
    // after the last one)
    const int flags = (sim < a.n_sims ? 1 : 0) | (sim == 0 ? 16 : 0);
    tree_phase<false, true, false>(a.s, sim - 1, a.ucb_table, a.discount, sc, flags, b_raw, half, tb);
    if (sim < a.n_sims) {
      __syncwarp();  // every lane's stores of the slice happen before lane 0's release
      if (lane == 0) tc::v4::red_release_add(pc.tree_done + (size_t)pair * 8, 1u);
    }
    if (stats) {
      const long long c2 = clock64();
      t_wait += c1 - c0;
      t_work += c2 - c1;
    }
  }
  if (stats) {
    atomicAdd(pc.stats + 0, (unsigned long long)t_wait);
    atomicAdd(pc.stats + 1, (unsigned long long)t_work);
    atomicAdd(pc.stats + 2, (unsigned long long)n_items);
    atomicAdd(pc.stats + 3, (unsigned long long)(clock64() - t_begin));
    atomicAdd(pc.stats + 7, 1ull);
  }
}

__global__ void __launch_bounds__(kPersistThreads, 1) search_persistent(const __grid_constant__ PersistArgs a) {
  extern __shared__ uint8_t smem_raw[];
  if ((int)blockIdx.x < a.n_mlp) {
    // all 24 warps: the body's roles use 22 of them, the two spare warps only take part in its block-wide barriers
    tc::v4::net_tc_body<false, true>(a.net, a.ctl, smem_raw, (int)blockIdx.x, a.n_mlp);
  } else {
    tree_role(a, smem_raw);
  }
}

// ---- server schedule (HMZ_SCHEDULE_SERVER): the MLP role alone stays resident (search_persistent launched with MLP CTAs
// only), the tree phases are ORDINARY launches of the fused kernel below on the remaining SMs, one per simulation and
// stream group.  Hand-off per 256-search tile pair, both ways through memory:
//   tree -> MLP   every warp adds 1 to tree_done[pair] (release) after its 16 searches' selection of simulation `sim`
//   MLP -> tree   mlp_done[pair] = sim (release) once the network outputs of simulation sim - 1 are stored; the warps of
//                 the tree launch for `sim` poll it before their backup (acquire)
// A network CTA needs a whole SM, so under the launch-per-simulation schedule the two kernel families take turns on the
// machine (DESIGN.md §4); here the network CTAs keep their SMs and the tree blocks never wait for an SM to drain.
static int server_mlp_ctas() {
  static const int v = getenv("HMZ_SERVER_MLP") ? atoi(getenv("HMZ_SERVER_MLP")) : 72;
  return v;
}

// Dynamic shared memory of search_persistent, opted in once per host thread and device.
static int persist_prepare(int* smem_out) {
  static thread_local int attr_dev = -1;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return fail(HMZ_ERR_CUDA, "cudaGetDevice failed");
  const int smem = (int)sizeof(tc::v4::Smem) + 1024;
  if (attr_dev != dev) {
    if (cudaFuncSetAttribute(search_persistent, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) != cudaSuccess)
      return fail(HMZ_ERR_CUDA, "cudaFuncSetAttribute(search_persistent): %s", cudaGetErrorString(cudaGetLastError()));
    attr_dev = dev;
  }
  *smem_out = smem;
  return HMZ_OK;
}

// The control block of both schedules for n_pairs tile pairs: ticket counter [0], queue tail [256], tree_done [1024, 32 B
// per pair), the item queue (8 B per slot, a power of two >= 2 n_pairs), then the server schedule's mlp_done (32 B per
// pair) and group_done (32 B per stream group, up to 16).  Returns its size in bytes; with `c`, also points c's hand-off
// words into `mem` — mlp_done and group_done only for the server schedule (with mlp_done set, the network body pushes no
// items to the queue).
static int64_t ctl_layout(int64_t n_pairs, void* mem, bool server, tc::v4::PersistCtl* c) {
  int64_t cap = 64;
  while (cap < 2 * n_pairs) cap <<= 1;
  const int64_t queue = 1024 + n_pairs * 32, mlp_done = queue + cap * 8 + 256, group_done = mlp_done + n_pairs * 32 + 256;
  if (c) {
    char* ctl = (char*)mem;
    c->tree_head = (uint32_t*)ctl;
    c->q_tail = (uint32_t*)(ctl + 256);
    c->tree_done = (uint32_t*)(ctl + 1024);
    c->queue = (unsigned long long*)(ctl + queue);
    c->q_mask = (uint32_t)(cap - 1);
    if (server) {
      c->mlp_done = (uint32_t*)(ctl + mlp_done);
      c->group_done = (uint32_t*)(ctl + group_done);
    }
  }
  return group_done + 768;
}

static int64_t tile_pairs(int64_t n_searches) { return (n_searches + 2 * tc::kM - 1) / (2 * tc::kM); }

// The MLP role's arguments: latents gathered from the leaf's parent record, written to record sim + 1 (the body derives
// the row).
static tc::v4::TcArgs mlp_args(const hmz_search_t* s, const void* weights, const TreeScratch& scratch, int n_pairs) {
  tc::v4::TcArgs a{};
  a.wsec = (const uint8_t*)weights;
  a.lat_in = s->latents;
  a.in_rows_per_item = s->n_records;
  a.in_row = scratch.leaf_parent;
  a.actions = scratch.leaf_action;
  a.lat_out = s->latents;
  a.out_rows_per_item = s->n_records;
  a.out_row = 0;
  a.latent_dtype = s->latent_dtype;
  a.r_out = const_cast<float*>(scratch.r);
  a.p_out = const_cast<float*>(scratch.p);
  a.v_out = const_cast<float*>(scratch.v);
  a.n = s->n_searches;
  a.n_pairs = n_pairs;
  return a;
}

// Launches the resident MLP CTAs on `mlp_stream`; the caller then enqueues the tree launches (server_tree_launch).
int server_mlp_launch(const hmz_search_t* s, const void* weights, int n_simulations, TreeScratch scratch, void* ctl_mem,
                      int pairs_per_group, cudaStream_t mlp_stream, ServerCtl* out) {
  int smem = 0;
  if (int rc = persist_prepare(&smem)) return rc;
  PersistArgs a{};
  a.n_pairs = (int)tile_pairs(s->n_searches);
  a.n_sims = n_simulations;
  int n_mlp = server_mlp_ctas();
  if (n_mlp > sm_count() - 8) n_mlp = sm_count() - 8;
  if (n_mlp > a.n_pairs) n_mlp = a.n_pairs;
  if (n_mlp < 1) return fail(HMZ_ERR_UNSUPPORTED, "server schedule needs at least 9 SMs");
  a.n_mlp = n_mlp;
  // (the caller has zeroed the control block and ordered every stream behind that)
  ctl_layout(a.n_pairs, ctl_mem, true, &a.ctl);
  a.ctl.n_sims = n_simulations;
  a.ctl.pairs_per_group = pairs_per_group;
  a.ctl.rotate = 1;
  a.net = mlp_args(s, weights, scratch, a.n_pairs);
  // tooling: HMZ_TC_TIMELINE=1 HMZ_TC_TIMELINE_PASS=p records the phase marks of CTA 0's pass p (hmz_debug_persist_timeline)
  a.net.timeline = (getenv("HMZ_TC_TIMELINE") && atoi(getenv("HMZ_TC_TIMELINE")))
                       ? (1 | ((getenv("HMZ_TC_TIMELINE_PASS") ? atoi(getenv("HMZ_TC_TIMELINE_PASS")) : 0) << 8))
                       : 0;
  search_persistent<<<dim3((unsigned)n_mlp), dim3(kPersistThreads), (size_t)smem, mlp_stream>>>(a);
  if (int rc = check_launch("search_persistent (server: MLP CTAs)")) return rc;
  out->tree_done = a.ctl.tree_done;
  out->mlp_done = a.ctl.mlp_done;
  out->group_done = a.ctl.group_done;
  return HMZ_OK;
}

static int persist_stats_on() {
  static const int v = getenv("HMZ_PERSIST_STATS") ? atoi(getenv("HMZ_PERSIST_STATS")) : 0;
  return v;
}
int persist_read_timeline(unsigned long long* host_out) {  // this translation unit's copy of the MLP body's phase marks
  return cudaMemcpyFromSymbol(host_out, tc::g_timeline, sizeof(unsigned long long) * 96) == cudaSuccess ? HMZ_OK : HMZ_ERR_CUDA;
}
int persist_read_stats(unsigned long long* host_out) {
  return cudaMemcpyFromSymbol(host_out, g_persist_stats, sizeof(unsigned long long) * 16) == cudaSuccess ? HMZ_OK : HMZ_ERR_CUDA;
}
static int persist_mlp_override() {
  static const int v = getenv("HMZ_PERSIST_MLP") ? atoi(getenv("HMZ_PERSIST_MLP")) : 0;
  return v;
}
static int persist_sm_limit() {
  static const int v = getenv("HMZ_PERSIST_SMS") ? atoi(getenv("HMZ_PERSIST_SMS")) : 0;
  return v;
}

// How many CTAs play the MLP role: the MLP side needs ceil(n_pairs / n_mlp) passes of ~8 us per simulation round, the
// tree side ~14 us per phase for as many slices as its 24 warps per CTA can hold at once; take the split that minimises
// the longer of the two (ties: fewer MLP CTAs).
static int choose_n_mlp(int n_pairs, int sms) {
  if (persist_mlp_override() > 0) return persist_mlp_override() < sms ? (persist_mlp_override() < n_pairs ? persist_mlp_override() : n_pairs) : sms - 1;
  const double t_mlp = 8.0, t_tree = 14.0;
  int best = 1;
  double best_cost = 1e30;
  for (int m = 1; m <= n_pairs && m < sms; ++m) {
    const int t = sms - m;
    const double mlp = (double)((n_pairs + m - 1) / m) * t_mlp;
    double tree = (double)n_pairs * tc::v4::kSlicesPerPair * t_tree / ((double)t * kPersistWarps);
    if (tree < t_tree) tree = t_tree;
    const double cost = mlp > tree ? mlp : tree;
    if (cost < best_cost - 1e-9) {
      best_cost = cost;
      best = m;
    }
  }
  return best;
}

int64_t persist_ctl_bytes(int64_t n_searches) { return ctl_layout(tile_pairs(n_searches), nullptr, false, nullptr); }

bool persist_supported(const hmz_search_t* s, int mode, int n_simulations) {
  return mode == HMZ_MODE_BF16 && n_simulations + 2 <= 2048 && s->n_searches > 0 && s->n_searches <= (int64_t)65535 * 256 &&
         n_simulations < 65535;
}

// scratch: the carved per-search arrays of hmz_search_run (p, r, v, leaf scalars, wild flags, path elements); ctl: zeroed
// here.  Returns HMZ_OK or an error; the caller has validated the descriptor (check_search) and the tables.
int persist_launch(const hmz_search_t* s, const void* weights, int n_simulations, const double* ucb_table, double discount,
                   const CountRow* cnt_table, const TreeScratch& scratch, void* ctl_mem, cudaStream_t stream) {
  int smem = 0;
  if (int rc = persist_prepare(&smem)) return rc;
  int sms = sm_count();
  if (persist_sm_limit() > 1 && persist_sm_limit() < sms) sms = persist_sm_limit();
  PersistArgs a{};
  const int64_t B = s->n_searches;
  a.n_pairs = (int)tile_pairs(B);
  a.n_sims = n_simulations;
  a.n_mlp = choose_n_mlp(a.n_pairs, sms);
  // every remaining SM plays the tree role, but never more CTAs than there are slices per simulation: with few searches
  // the slices spread one or two per SM (a warp alone on its scheduler runs its dependent chain fastest); warps that
  // find no ticket left exit at once
  const int tree_want = a.n_pairs * tc::v4::kSlicesPerPair;
  int n_tree = sms - a.n_mlp;
  if (n_tree > tree_want) n_tree = tree_want;
  if (n_tree < 1) return fail(HMZ_ERR_UNSUPPORTED, "persistent search needs at least 2 SMs");
  a.table_rows = n_simulations + 2;
  if ((size_t)a.table_rows * (sizeof(CountRow) + sizeof(double)) + 256 > (size_t)smem)
    return fail(HMZ_ERR_UNSUPPORTED, "persistent search: %d simulations exceed the shared-memory tables", n_simulations);
  a.total_tickets = (uint32_t)tc::v4::kSlicesPerPair * (uint32_t)a.n_pairs * (uint32_t)(n_simulations + 1);
  a.s = *s;
  a.cnt_table = cnt_table;
  a.ucb_table = ucb_table;
  a.discount = discount;
  a.sc = scratch;
  a.sc.capture = s->capture;
  a.capture_stride = s->capture ? B * 8 : 0;
  const int64_t ctl_bytes = ctl_layout(a.n_pairs, ctl_mem, false, &a.ctl);
  if (cudaMemsetAsync(ctl_mem, 0, (size_t)ctl_bytes, stream) != cudaSuccess) return fail(HMZ_ERR_CUDA, "cudaMemsetAsync(control block) failed");
  a.ctl.n_sims = n_simulations;
  if (tc::v4::kPersistStats && persist_stats_on()) {
    void* sp = nullptr;
    if (cudaGetSymbolAddress(&sp, g_persist_stats) != cudaSuccess || cudaMemsetAsync(sp, 0, sizeof(unsigned long long) * 16, stream) != cudaSuccess)
      return fail(HMZ_ERR_CUDA, "persistent search: statistics buffer unavailable");
    a.ctl.stats = (unsigned long long*)sp;
  }
  a.net = mlp_args(s, weights, scratch, a.n_pairs);
  void* params[] = {&a};
  const cudaError_t e = cudaLaunchCooperativeKernel((const void*)search_persistent, dim3((unsigned)(a.n_mlp + n_tree)), dim3(kPersistThreads),
                                                    params, (size_t)smem, stream);
  if (e != cudaSuccess) return fail(HMZ_ERR_CUDA, "search_persistent launch (%d MLP + %d tree CTAs): %s", a.n_mlp, n_tree, cudaGetErrorString(e));
  return check_launch("search_persistent");
}

}  // namespace hmz
