/* hmz.h — C ABI of libhmz.so, the B200-native batched MuZero/Hanoi acting engine.
 *
 * This header is the drop-in boundary for ONE hot path of A-Andrews/Muzero-Hanoi:
 *   Hanoi env step -> MCTS select / expand / backup -> dynamics+prediction MLP ->
 *   root visit histogram -> action sampling.
 * The reference has no FFI layer (it is pure Python); each entry point below therefore
 * names the reference *Python function* it replaces (file:line under the reference
 * repository), and INTEGRATION.md shows the ctypes binding a maintainer would add.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes only; no torch / C++ types cross the boundary.
 *   - Every pointer is a DEVICE pointer owned by the caller unless the name says `host_`.
 *   - The library never allocates device memory and never synchronises: kernels are
 *     enqueued on `stream` (a cudaStream_t passed as void*, NULL = legacy default stream).
 *   - Every function returns HMZ_OK (0) or a negative HMZ_ERR_* code and never throws;
 *     hmz_last_error() returns a thread-local message for the last failure.
 *   - Re-entrant per descriptor: results depend only on the arguments of a call.  Process-wide state is
 *     limited to the thread-local error string, the launch counter (hmz_launch_count), lazily created
 *     per-thread helper streams / constant tables, and the TOOLING hooks hmz_prof_* / hmz_debug_* (one
 *     profiling session per process at a time); none of it changes what a call computes.
 *   - There is NO CPU fallback: without a CUDA device every compute entry point fails
 *     with HMZ_ERR_CUDA.
 */
#ifndef HMZ_H
#define HMZ_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HMZ_OK 0
#define HMZ_ERR_INVALID (-1)     /* bad argument (size, range, null pointer)            */
#define HMZ_ERR_CUDA (-2)        /* CUDA runtime / launch error                          */
#define HMZ_ERR_UNSUPPORTED (-3) /* valid request this build cannot serve (e.g. N > 12)  */

#define HMZ_N_ACTIONS 6  /* env/hanoi.py:39-41: permutations(range(3), 2)               */
#define HMZ_LATENT 64    /* networks.py:22  reprs_output_size                            */
#define HMZ_HIDDEN 256   /* networks.py:21  h1_s                                         */
#define HMZ_SUPPORT 33   /* networks.py:34-35 support_size when TD_return=True           */
#define HMZ_MAX_DISKS 12 /* 2 bits/disk + >= 8 counter bits in one 32-bit env word       */
#define HMZ_NO_CHILD 0xFFFFu

/* flag bits written by hmz_env_step* (one uint8 per env) */
#define HMZ_FLAG_DONE 1u    /* env/hanoi.py:68,78  done                                   */
#define HMZ_FLAG_ILLEGAL 2u /* env/hanoi.py:54     illegal_move                           */
#define HMZ_FLAG_GOAL 4u    /* env/hanoi.py:65-69  goal reached (reward 100)              */
#define HMZ_FLAG_TRUNC 8u   /* env/hanoi.py:77-80  step_counter == max_steps              */

const char* hmz_last_error(void);
int hmz_version(void);
/* Names of the non-default compile-time tuning switches this library was built with ("" = the shipped
 * configuration).  None of them changes results; tests assert a clean build. */
const char* hmz_build_flags(void);
/* Number of kernels this library has launched from the calling process (for bench.py's
 * gpu_launches claim). */
int64_t hmz_launch_count(void);
int hmz_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* Optional per-kernel timing for bench.py's roofline: between hmz_prof_begin() and
 * hmz_prof_end() every kernel this library launches is bracketed by a CUDA-event pair on its
 * own stream.  hmz_prof_end synchronises those events and returns, per kernel class, the summed
 * device time in milliseconds and the number of launches.  Classes: */
#define HMZ_PROF_ENV 0
#define HMZ_PROF_SELECT 1
#define HMZ_PROF_NET_RECURRENT 2
#define HMZ_PROF_EXPAND_BACKUP 3
#define HMZ_PROF_NET_INITIAL 4
#define HMZ_PROF_ROOT_POLICY 5
#define HMZ_PROF_OTHER 6
#define HMZ_PROF_SEARCH_PERSISTENT 7 /* the one-launch-per-move search kernel (HMZ_SCHEDULE_PERSISTENT) */
#define HMZ_PROF_CLASSES 8
int hmz_prof_begin(void);
int hmz_prof_end(double* ms_by_class, int64_t* launches_by_class);

/* ------------------------------------------------------------------ environment ----
 * Env word (uint32): bits [0, 2N) hold the peg (0..2) of disk d at bits [2d, 2d+2), disk 0
 * smallest — the tuple of env/hanoi.py:19-25 packed; bits [2N, 32) hold step_counter
 * (env/hanoi.py:45,56).  Requires N <= HMZ_MAX_DISKS and max_steps < 2^(32-2N).
 */

/* words[i] = reset_word for all i (TowersOfHanoi.reset, env/hanoi.py:86-96). */
int hmz_env_reset(uint32_t* words, int64_t n_envs, uint32_t reset_word, void* stream);

/* words[i] = packed state of states[index[i]] where the index is the base-3 number with
 * disk 0 as most significant digit (itertools.product order, env/hanoi.py:23-25).  Used by
 * random_reset (env/hanoi.py:98-111) with host-drawn indices in parity mode. */
int hmz_env_from_index(const uint32_t* index, uint32_t* words, int64_t n_envs, int n_disks, void* stream);
int hmz_env_to_index(const uint32_t* words, uint32_t* index, int64_t n_envs, int n_disks, void* stream);

/* TowersOfHanoi.random_reset drawn on device: uniform over the 3^N - 1 non-goal states,
 * Philox4x32-10 keyed by (seed, env id, counter). */
int hmz_env_random_reset(uint32_t* words, int64_t n_envs, int n_disks, int goal_peg, uint64_t seed,
                         uint64_t counter, void* stream);

/* TowersOfHanoi.step (env/hanoi.py:47-84) for n_envs envs at once.
 *   words    in/out  env words (state + counter)
 *   actions  in      action index 0..5 per env
 *   rewards  out     0.0f, 100.0f or -0.1f  (env/hanoi.py:62,66,72)
 *   flags    out     HMZ_FLAG_* bits
 *   obs_words out, nullable: packed state the returned observation encodes (the GOAL state
 *            when the goal is reached although the stored state is not updated, :65-69)
 *   auto_reset != 0: envs that finish are set to reset_word (counter 0) in the same pass.
 *   auto_reset == 0: finished envs keep the reference's stored state with counter 0; the
 *            caller must reset them before stepping again (env/hanoi.py:49).
 */
int hmz_env_step(uint32_t* words, const uint8_t* actions, float* rewards, uint8_t* flags, uint32_t* obs_words,
                 int64_t n_envs, int n_disks, int max_steps, int goal_peg, int auto_reset, uint32_t reset_word,
                 void* stream);

/* Bit a of mask[i] = TowersOfHanoi._move_allowed(moves[a]) (env/hanoi.py:123-139). */
int hmz_env_legal_mask(const uint32_t* words, uint8_t* mask, int64_t n_envs, int n_disks, void* stream);

/* utils.oneHot_encoding (utils.py:9-25) as float32 [n_envs, 3N], disk-major. */
int hmz_env_onehot(const uint32_t* words, float* obs, int64_t n_envs, int n_disks, void* stream);

/* env.hanoi_utils.hanoi_solver (env/hanoi_utils.py:4-26): minimal moves to goal_peg. */
int hmz_env_solver_distance(const uint32_t* words, uint32_t* distance, int64_t n_envs, int n_disks, int goal_peg,
                            void* stream);

/* One env step with a uniformly random LEGAL move drawn on device (BASELINE.json config 4;
 * the host equivalent scans _move_allowed over moves as legal_illegal_preds.py:51 does).
 * Writes the chosen action, reward and flags (13 B / env step of traffic). */
int hmz_env_step_random(uint32_t* words, uint8_t* actions, float* rewards, uint8_t* flags, int64_t n_envs,
                        int n_disks, int max_steps, int goal_peg, uint32_t reset_word, uint64_t seed,
                        uint64_t step_index, void* stream);

/* n_steps random-legal-move steps per env fused in registers (state read and written once).
 * counters (device, uint64[4], accumulated with atomics): [0] steps taken, [1] goals reached,
 * [2] truncations, [3] xor-fold checksum of final words.  Auto-resets to reset_word. */
int hmz_env_rollout_random(uint32_t* words, int64_t n_envs, int n_disks, int max_steps, int goal_peg,
                           uint32_t reset_word, int n_steps, uint64_t seed, uint64_t step_index,
                           unsigned long long* counters, void* stream);

/* ------------------------------------------------------------------ tree store -----
 * One 128-byte record per EXPANDED node = two 64-byte halves, each holding three child slots
 * (one 16-byte slot per child action: W, rwd, N, child record) followed by those children's
 * priors.  A search is owned by a pair of lanes; each lane's whole share of a pUCT decision is
 * its 64-byte half (four 128-bit loads), and a backup step is one 16-byte slot read + write.
 * The node expanded by simulation s of a search is record s+1 (root = record 0), so no
 * allocator is needed.  Fields restate MCTS/node.py:9-28 (prior, N, W, rwd, children).
 */
typedef struct hmz_child {
  double W;       /* child.W   (float64 sum of backed-up values, node.py:63)              */
  float rwd;      /* child.rwd  (float32 value, widened exactly when used)                */
  uint16_t N;     /* child.N                                                              */
  uint16_t child; /* record index of the expanded child, HMZ_NO_CHILD otherwise           */
} hmz_child_t;

typedef struct hmz_half {
  hmz_child_t c[3];      /* children 3h .. 3h+2 of the node                               */
  float prior[3];        /* their priors (float32; a noised root keeps float64 in root_prior) */
  uint16_t parent;       /* half 0 only: record index of this node's parent (root: 0)     */
  uint8_t parent_action; /* half 0 only: action that leads from the parent to this node   */
  uint8_t pad;
} hmz_half_t;

typedef struct hmz_node {
  hmz_half_t h[2]; /* child a lives in h[a / 3].c[a % 3], its prior in h[a / 3].prior[a % 3] */
} hmz_node_t;

#define HMZ_LATENT_F32 0
#define HMZ_LATENT_BF16 1

typedef struct hmz_search {
  hmz_node_t* nodes;   /* [n_searches][n_records]                                        */
  void* latents;       /* [n_searches][n_records][64] float32 or bf16 (node.h_state)     */
  double* root_prior;  /* [n_searches][6] float64 root priors (exact copy of the input)   */
  double* root_W;      /* [n_searches]   root.W                                           */
  double* minmax;      /* [n_searches][2] (min, max) of MinMaxStats; PERSISTS across calls */
  void* workspace;     /* hmz_search_workspace_bytes(n_searches) bytes of scratch          */
  float* capture;      /* nullable [n_simulations][n_searches][8]: hmz_search_run records the network outputs
                          p[6], r, v of every simulation here (parity tests replay them through the oracle) */
  int64_t n_searches;
  int32_t n_records;   /* >= n_simulations + 1                                           */
  int32_t latent_dtype;
  int32_t root_prior_is_f64; /* 1: noised root, U = f32(f64 prior * w) (node.py:122)      */
  int32_t schedule;    /* hmz_search_run scheduling, never changes results: 0 = automatic; k in [1, 16] = one
                          launch pair per simulation with the batch cut into k concurrent stream groups;
                          HMZ_SCHEDULE_PERSISTENT = one persistent role-specialised kernel per call;
                          HMZ_SCHEDULE_SERVER | k = network CTAs resident for the whole call on a fixed share of the
                          SMs, fed through memory flags by ordinary tree-kernel launches in k stream groups (0: 4) */
} hmz_search_t;
#define HMZ_SCHEDULE_AUTO 0
#define HMZ_SCHEDULE_PERSISTENT 64
#define HMZ_SCHEDULE_SERVER 128

/* Scratch needed by hmz_search_run (per-simulation leaf ids and network outputs). */
int64_t hmz_search_workspace_bytes(int64_t n_searches);

/* MinMaxStats() construction (MCTS/utils_mcts.py:4-6): (min, max) = (+inf, -inf). */
int hmz_search_minmax_reset(double* minmax, int64_t n_searches, void* stream);

/* root_node.expand(prior, h, 0.0) (MCTS/mcts.py:52-69): clears record 0, stores priors.
 * The root latent must already be in latents[:, 0, :] (written by hmz_net_initial). */
int hmz_search_begin(const hmz_search_t* s, const double* root_prior, void* stream);

/* Same, with the root prior built on the device from the float32 policy p0 [n_searches][6] of
 * hmz_net_initial: prior = p0 when noise == NULL; otherwise add_dirichlet_noise
 * (MCTS/mcts.py:132-152) with the Dirichlet draw supplied as noise float64 [n_searches][6]:
 * prior = float64(float32(1-eps) * p0) + eps * noise.  s->root_prior_is_f64 must be
 * (noise != NULL). */
int hmz_search_begin_p0(const hmz_search_t* s, const float* p0, const double* noise, double eps, void* stream);

/* Phase 1 of one simulation (MCTS/mcts.py:75-86 -> Node.best_child, node.py:72-123) for all
 * searches: walk from the root taking arg-max of f32(Q)+f32(U) (lowest index on ties) until an
 * unexpanded child.  ucb_table[n] = (log((n+19653)/19652)+1.25)*sqrt(n) for n in [0, sim],
 * float64, computed by the host libm exactly as node.py:114-120 does.
 *   leaf_parent/leaf_action/leaf_depth out: record of the leaf's parent, its action, path length
 *   path_out nullable [n_searches][path_cap]: actions root->leaf (0xFF padded), diagnostics. */
int hmz_search_select(const hmz_search_t* s, int sim, const double* ucb_table, double discount,
                      uint16_t* leaf_parent, uint8_t* leaf_action, uint16_t* leaf_depth, uint8_t* path_out,
                      int path_cap, void* stream);

/* Node.child_Q and Node.child_U (MCTS/node.py:90-123) of one expanded node per search, for
 * inspection through the Node view: record[i] names the node, node_n[i] is that node's own visit
 * count (the N that enters the exploration factor).  q_out, u_out float32 [n_searches][6];
 * best_out (nullable) = Node.best_child's arg-max of q+u with lowest-index tie-break. */
int hmz_search_child_scores(const hmz_search_t* s, const uint16_t* record, const int32_t* node_n, const double* ucb_table,
                            double discount, float* q_out, float* u_out, int32_t* best_out, void* stream);

/* Phases 2b+3 (MCTS/mcts.py:106-109 -> Node.expand node.py:30-51, Node.backup :53-70) with the
 * network outputs of this simulation given per search: creates record sim+1 with priors p,
 * stores r on the leaf slot, then walks to the root: W += value; N += 1;
 * minmax.update(rwd + discount*Q); value = rwd + discount*value — all float64. */
int hmz_search_expand_backup(const hmz_search_t* s, int sim, double discount, const uint16_t* leaf_parent,
                             const uint8_t* leaf_action, const float* r, const float* p, const float* v,
                             void* stream);

/* MCTS/mcts.py:112-126: child_N, generate_play_policy (:154-176), arg-max or sampled action.
 *   uniforms nullable unless deterministic == 0 (one double in [0,1) per search; the draw of
 *   np.random.choice at :120 supplied as input);  outputs nullable individually.
 *   pow_table nullable: float64 [n_simulations + 1][6], pow_table[n][a] = element a of
 *   np.power(int64 array of six n, clamp(1/T, 1, 5)) as the caller's NumPy evaluates it (:170-174).  NumPy's
 *   vectorised pow is not correctly rounded and differs between its SIMD body and its scalar tail (so by
 *   position in the 6-element array) and between CPUs; bit-exact policies for non-integer exponents (or powers
 *   beyond 2^53) therefore need the caller's own table.  NULL: the device evaluates integer exponents by exact
 *   repeated multiplication (identical to NumPy while the power stays below 2^53, i.e. counts < 1,552 at
 *   exponent 5) and others with CUDA's pow() (<= 2 ulp). */
int hmz_search_root_policy(const hmz_search_t* s, int n_simulations, double temperature, int deterministic,
                           const double* uniforms, const double* pow_table, int32_t* visits, double* pi, double* root_q,
                           int32_t* action, void* stream);

/* ------------------------------------------------------------------ networks -------
 * Packed weights: one device blob produced by hmz_weights_pack from the 20 tensors of
 * MuZeroNet.state_dict() (networks.py:39-67), in the order
 *   {representation_net, dynamic_net, rwd_net, policy_net, value_net} x {0.weight, 0.bias,
 *   2.weight, 2.bias}.
 */
#define HMZ_MODE_FP32 0 /* FFMA, fp32 accumulate: parity mode (<= 1e-5 vs reference)      */
#define HMZ_MODE_BF16 1 /* tcgen05 bf16 x bf16 -> fp32 in TMEM: throughput mode (<= 2e-2) */
#define HMZ_MODE_FP32X3 2 /* fast parity mode: the network on tcgen05 with every float32 operand split into three
                           * bf16 parts (7 exact bf16 products per multiply, fp32 accumulate; <= 1e-5 vs reference, same gate
                           * as HMZ_MODE_FP32), for both inferences from packed env words; float observations (hmz_net_initial with obs) run the
                           * FFMA kernel on an embedded float32 copy */

int64_t hmz_weights_packed_bytes(int n_disks, int mode);
/* host_tensors: 20 HOST pointers to contiguous float32 tensors; host_out: HOST buffer of
 * hmz_weights_packed_bytes() bytes that the caller then copies to the device. */
int hmz_weights_pack(const float* const* host_tensors, int n_disks, int mode, void* host_out);

/* MuZeroNet.initial_inference (networks.py:71-94) for a batch of packed env words:
 * h0 = normalize(representation_net(onehot(word))), p0 = softmax(policy_net(h0)),
 * v0 = support_to_scalar(value_net(h0)).  h0 row i is written to
 * latents_out + (i*out_rows_per_item)*64 elements (so it can target record 0 of a search). */
int hmz_net_initial(const void* weights, int mode, int n_disks, const uint32_t* words, const float* obs,
                    void* latents_out, int64_t out_rows_per_item, int latent_dtype, float* p0, float* v0,
                    int64_t n, void* stream);

/* MuZeroNet.recurrent_inference (networks.py:96-116) for a batch:
 * input latent of item i  = latents_in  + (i*in_rows_per_item  + in_row[i]) * 64   (in_row nullable = 0)
 * output latent of item i = latents_out + (i*out_rows_per_item + out_row)   * 64
 * r, v float32 [n]; p float32 [n,6] (softmax probabilities). */
int hmz_net_recurrent(const void* weights, int mode, const void* latents_in, int64_t in_rows_per_item,
                      const uint16_t* in_row, const uint8_t* actions, void* latents_out,
                      int64_t out_rows_per_item, int64_t out_row, int latent_dtype, float* r, float* p, float* v,
                      int64_t n, void* stream);

/* Whole search, fused: n_simulations x (select -> g+f MLP -> expand -> backup) for every
 * search in one launch sequence with no host round trips (MCTS.run_mcts, MCTS/mcts.py:71-109). */
int hmz_search_run(const hmz_search_t* s, const void* weights, int mode, int n_simulations,
                   const double* ucb_table, double discount, void* stream);
/* (Scheduling is chosen per call by hmz_search_t.schedule.) */

/* ------------------------------------------------------------------ heterogeneous batches ---
 * One search batch over several networks and simulation budgets (the lesion-experiment grid of
 * acting_ablations.get_results run as one batch).  The batch is cut into blocks of 256 searches:
 *   - every block uses ONE weight set: sets are packed (hmz_weights_pack, same n_disks and mode) into one
 *     device blob at a fixed stride, set k at weights + k * weight_stride;
 *   - every search has its own budget, in [1, host_block_budget[its block]];
 *   - blocks are ordered by non-increasing budget, so simulation s runs over a prefix of the batch: the
 *     blocks whose budget is greater than s.
 * A search with budget b runs simulations 0 .. b-1 exactly as hmz_search_run with n_simulations = b
 * would run it alone; its node records and latents above record b are unspecified afterwards. */
typedef struct hmz_multi {
  const uint16_t* block_set;         /* device [n_searches / 256]: weight set of each block, in [0, n_sets)       */
  const uint16_t* budget;            /* device [n_searches]: simulations of each search (nullable for initial) */
  const int32_t* host_block_budget;  /* HOST [n_searches / 256]: max budget of each block, non-increasing        */
  int64_t weight_stride;             /* bytes between sets: >= hmz_weights_packed_bytes, a multiple of 256      */
  int32_t n_sets;                    /* weight sets in the blob (>= 1)                                          */
  int32_t n_disks;                   /* disk count the sets were packed for                                     */
} hmz_multi_t;

/* hmz_net_initial from packed env words with each block's weight set (n = n_searches of m, a multiple of 256;
 * host_block_budget and budget are not read). */
int hmz_net_initial_multi(const void* weights, const hmz_multi_t* m, int mode, const uint32_t* words, void* latents_out,
                          int64_t out_rows_per_item, int latent_dtype, float* p0, float* v0, int64_t n, void* stream);
/* hmz_search_run over a heterogeneous batch: simulation s launches the select -> MLP -> backup chain over the
 * blocks whose budget is greater than s; within them a search backs up simulation s only if s < budget and
 * selects the next leaf only if s + 1 < budget.  s->n_records >= host_block_budget[0] + 1.  Schedules: 0 and
 * k in [1, 16] (stream groups of whole blocks); HMZ_SCHEDULE_PERSISTENT / _SERVER: HMZ_ERR_UNSUPPORTED. */
int hmz_search_run_multi(const hmz_search_t* s, const hmz_multi_t* m, const void* weights, int mode, const double* ucb_table,
                         double discount, void* stream);
/* hmz_search_root_policy with root_q = root_W / budget[b] per search; pow_table (nullable) has
 * host_block_budget[0] + 1 rows. */
int hmz_search_root_policy_multi(const hmz_search_t* s, const hmz_multi_t* m, double temperature, int deterministic,
                                 const double* uniforms, const double* pow_table, int32_t* visits, double* pi, double* root_q,
                                 int32_t* action, void* stream);

/* Tooling only: with HMZ_TC_TIMELINE=1 in the environment, CTA 0 of the tensor-core kernel records
 * clock64() at its phase boundaries; this copies the 96 marks of the last launch to the host. */
int hmz_debug_tc_timeline(unsigned long long* host_out);
/* Tooling only: the same for the HMZ_MODE_FP32X3 kernel (HMZ_X3_TIMELINE=1): 160 marks of CTA 0's first tile — [g] / [16 + g]
 * first layer of chunk g issued from / to, [32 + g] / [48 + g] second layer, [64 + g] / [80 + g] hidden epilogue of chunk g
 * (epilogue thread 0), [96 + net] / [100 + net] output epilogue of a network, [106] raw latent tile published, [104] / [105] gather, [110] / [111] prologue,
 * [112 + g] first-layer warp at its loop top, [128 + g] first-layer weight block's TMA issued, [144 + g] seen landed. */
int hmz_debug_x3_timeline(unsigned long long* host_out);
/* Tooling only: key = search | (simulation << 32) >= 0 switches hmz_search_run to the instrumented fused
 * backup + select kernel, whose lane pair `search` records clock64() at its phase boundaries in that
 * simulation (-1 switches it off); host_out (nullable, 64 values) receives the marks. */
int hmz_debug_tree_timeline(long long search, unsigned long long* host_out);
/* Tooling only: with HMZ_PERSIST_STATS=1 in the environment the persistent search kernel accumulates clock64 sums of its
 * last launch; host_out receives 16 values: [0] tree warps waiting for work, [1] tree warps working, [2] slices processed,
 * [3] summed tree-warp lifetimes, [4] MLP CTAs waiting for the tree (one thread each), [5] MLP CTAs first -> last hand-off,
 * [6] MLP passes, [7] tree warps. */
int hmz_debug_persist_stats(unsigned long long* host_out);
/* Tooling: clock64 phase marks (96 words) of MLP CTA 0 of the persistent / server schedules for the pass named by
 * HMZ_TC_TIMELINE=1 HMZ_TC_TIMELINE_PASS=p (same slots as hmz_debug_tc_timeline). */
int hmz_debug_persist_timeline(unsigned long long* host_out);
/* Tooling: launch Gantt of the hot-loop kernels.  enable = 1 starts recording; enable = 0 stops, synchronises the device
 * and writes up to max_records records of four words {kind (0 = network kernel, 1 = fused tree kernel), tag = sim << 8 |
 * group, first block's start, last block's end} (globaltimer ns) to host_out; *n_out = records written. */
int hmz_debug_gantt(int enable, unsigned long long* host_out, int max_records, int* n_out);
/* Tests only: compares the search kernels' exact-division shortcuts (table / precomputed reciprocal + two
 * FMA corrections) with IEEE division bit for bit on n_samples random operand pairs; adds the number of
 * mismatches to counters[0] (division by a visit count) and counters[1] (division by the min-max range). */
int hmz_debug_div_check(uint64_t n_samples, uint64_t seed, unsigned long long* counters, void* stream);

/* ------------------------------------------------------------------ self-play glue ---
 * Throughput-mode randomness, drawn on device with Philox4x32-10 keyed by (seed, GLOBAL item id, counter): item i of
 * a call is keyed by item_offset + i, so results do not depend on how games are sharded over GPUs (rank r of G passes
 * the global id of its first game).  Parity mode passes the reference's own draws to hmz_search_begin_p0 /
 * hmz_search_root_policy instead.
 */
/* np.random.dirichlet(alpha * ones(6)) (MCTS/mcts.py:148-149): out float64 [n][6].  counter < 2^56
 * (HMZ_ERR_INVALID otherwise): the gamma streams keep the draw's block number in the low 8 bits of Philox counter
 * word 3, so counter bits 56-63 have no room there. */
int hmz_rng_dirichlet(double* out, int64_t n, double alpha, uint64_t seed, uint64_t counter, uint64_t item_offset, void* stream);
/* One uniform double in [0, 1) per item (the draw of np.random.choice, MCTS/mcts.py:120). */
int hmz_rng_uniform(double* out, int64_t n, uint64_t seed, uint64_t counter, uint64_t item_offset, void* stream);
/* The same draw with its key given per item: out[i] = the uniform of item item[i] at counter counter_hi[i] | counter_lo,
 * i.e. element item[i] - o of hmz_rng_uniform(seed, counter_hi[i] | counter_lo, item_offset o).  Items of different
 * streams (a batch of several experiments) draw in one launch. */
int hmz_rng_uniform_keyed(double* out, int64_t n, uint64_t seed, const uint64_t* counter_hi, uint64_t counter_lo,
                          const uint64_t* item, void* stream);
/* Tests only: n_blocks raw Philox4x32-10 blocks; counters_keys uint32 [n_blocks][6] = counter words 0..3, key words
 * 0..1; out uint32 [n_blocks][4] (known-answer vectors of Salmon et al. 2011). */
int hmz_debug_philox(const uint32_t* counters_keys, uint32_t* out, int n_blocks, void* stream);

/* One game-move — the episode lists of Muzero._play_game (Muzero.py:179-183) for one step — as a 32-byte record:
 * the element of the trajectory ring AND the wire format of the NCCL all-gather towards the replay buffer. */
typedef struct hmz_move_record {
  double root_q;      /* root_node.Q (float64, so n-step returns computed downstream stay bit-exact)   */
  uint32_t state;     /* env word BEFORE the move                                                      */
  float reward;       /* 0, 100 or -0.1 (env/hanoi.py:62,66,72)                                        */
  uint16_t visits[6]; /* root child visit counts                                                       */
  uint8_t action;     /* sampled action                                                                */
  uint8_t flags;      /* HMZ_FLAG_* of the move                                                        */
  uint16_t game_lo;   /* low 16 bits of the global game id (ordering check after a gather)             */
} hmz_move_record_t;

/* One move of every game, fused on the host side of the ABI (the `hmz_selfplay_round` of SURVEY.md §8b): the loop body
 * of Muzero._play_game (Muzero.py:165-186) for all games — hmz_net_initial; ONE kernel for the Dirichlet draw, its mix
 * into the root prior (hmz_search_begin_p0) and the sampling uniform, keyed by (seed, game_offset + game, move_index);
 * hmz_search_run; ONE kernel for the root policy + sampled action (hmz_search_root_policy), the move record, the
 * episode store (hmz_episode_record / _close) and hmz_env_step with auto-reset — enqueued on `stream` without any host
 * synchronisation.  All pointers are caller-owned device buffers.  move_index < 2^56 (HMZ_ERR_INVALID otherwise), the
 * counter domain of hmz_rng_dirichlet. */
typedef struct hmz_selfplay {
  hmz_search_t search;      /* root_prior_is_f64 must equal (dirichlet_alpha > 0 && exploration_eps > 0) */
  const void* weights;      /* hmz_weights_pack blob */
  const double* ucb_table;  /* as hmz_search_select */
  uint32_t* words;          /* [B] env words (stepped in place) */
  float* p0;                /* [B][6] root policy */
  float* v0;                /* [B] root value */
  double* noise;            /* [B][6] receives the Dirichlet draws (nullable) */
  double* uniform;          /* [B] receives the sampling uniforms */
  int32_t* visits;          /* [B][6] root child visit counts of the move (nullable) */
  double* root_q;           /* [B] root_node.Q (nullable) */
  int32_t* action;          /* [B] sampled action (nullable) */
  hmz_move_record_t* records; /* [B] this move's slot of the trajectory ring (nullable), 16-byte aligned */
  uint32_t* ep_state;       /* episode store (hmz_episode_record / _close), all NULL to skip */
  uint8_t* ep_action;
  uint8_t* ep_flags;
  uint16_t* ep_visits;
  double* ep_root_q;
  int32_t* ep_cur_slot;
  int32_t* ep_len;
  uint8_t* ep_exp;          /* nullable: receives the move's integer play-policy exponent (see hmz_episode_unroll) */
  const double* pow_table;  /* as hmz_search_root_policy (nullable) */
  double discount, dirichlet_alpha, exploration_eps, temperature;
  uint64_t seed;
  uint64_t game_offset;     /* global id of game 0 of this batch (Philox key, record.game_lo) */
  int32_t mode, n_disks, max_steps, goal_peg, n_simulations, ep_t_max;
  uint32_t reset_word;
  int32_t reserved;
} hmz_selfplay_t;
int hmz_selfplay_move(const hmz_selfplay_t* sp, uint64_t move_index, void* stream);

/* ------------------------------------------------------------------ episode post-processing ---
 * The tail of Muzero._play_game (Muzero.py:189-205) and Buffer.add (buffer.py:47-83) on the device.
 * Episode store: struct-of-arrays [t_max][n_games], slot = the game's own step counter (the counter
 * bits of its env word before the move), so slots [0, ep_len[g]) hold game g's current episode:
 *   ep_state u32 env word before the move | ep_action u8 | ep_flags u8 HMZ_FLAG_* of the move (the
 *   reward 0 / 100 / -0.1 is a function of them) | ep_visits u16[6] | ep_root_q f64 (root_node.Q).
 */
/* The episode lists of one move (Muzero.py:179-183) for every game; cur_slot[g] <- slot written. */
int hmz_episode_record(const uint32_t* words, const int32_t* action, const int32_t* visits, const double* root_q, int n_disks,
                       int t_max, int64_t n_games, uint32_t* ep_state, uint8_t* ep_action, uint16_t* ep_visits,
                       double* ep_root_q, int32_t* cur_slot, uint8_t* action_u8_out, void* stream);
/* After hmz_env_step: the move's flags join its slot; ep_len[g] = episode length if the game just
 * finished (HMZ_FLAG_DONE), else 0. */
int hmz_episode_close(const uint8_t* flags, const int32_t* cur_slot, int64_t n_games, uint8_t* ep_flags, int32_t* ep_len,
                      void* stream);
/* The episode store filled from move records, e.g. the all-gather of every rank's move: exactly the ep_* writes of
 * hmz_selfplay_move, for n_games records, record i being global game game_offset + i.  slot = the counter bits of
 * record.state (clamped to t_max - 1); state / action / flags / visits / root_q are stored there, cur_slot[i] = slot,
 * ep_len[i] = slot + 1 if HMZ_FLAG_DONE else 0, ep_exp (nullable) = the integer play-policy exponent clamp(1/T, 1, 5) of
 * `temperature` (HMZ_ERR_UNSUPPORTED if it is not an integer).  A record whose game_lo != (game_offset + i) & 0xFFFF
 * writes nothing and adds 1 to *mismatch (device int32).  records 16-byte aligned. */
int hmz_episode_ingest(const hmz_move_record_t* records, int64_t n_games, uint64_t game_offset, int n_disks, int t_max,
                       double temperature, uint32_t* ep_state, uint8_t* ep_action, uint8_t* ep_flags, uint16_t* ep_visits,
                       double* ep_root_q, int32_t* cur_slot, int32_t* ep_len, uint8_t* ep_exp, int32_t* mismatch, void* stream);
/* compute_n_step_returns (utils.py:28-72) and the priorities |f32(return) - f32(rootQ)|
 * (Muzero.py:197-200) of every finished episode (ep_len[g] > 0): returns float64 / priority float32
 * [t_max][n_games].  discount_pow[i] = discount ** i for i in [0, n_step], computed by the HOST libm
 * as the reference does; the discounted reward sum reproduces CPython's compensated float sum(). */
int hmz_episode_returns(const uint8_t* ep_flags, const double* ep_root_q, const int32_t* ep_len, int64_t n_games, int t_max,
                        const double* discount_pow, int n_step, double* returns, float* priority, void* stream);
/* compute_MCreturns (utils.py:75-86), the TD_return = False branch of Muzero._play_game (:193-194), with the same
 * outputs as hmz_episode_returns.  discount_pow[i] = discount ** i for i in [0, t_max) as NumPy's power ufunc
 * evaluates it on the host (the reference computes `discount ** np.array(range(T))`). */
int hmz_episode_mc_returns(const uint8_t* ep_flags, const double* ep_root_q, const int32_t* ep_len, int64_t n_games, int t_max,
                           const double* discount_pow, double* returns, float* priority, void* stream);
/* Replay rows of the finished episodes: row_base[g] = ptr + exclusive prefix sum of the stored lengths
 * (or -1), *total_out = rows to add.  only_solved != 0 keeps an episode only if returns[-1] > 0
 * (training_loop, Muzero.py:98). */
int hmz_episode_rows(const int32_t* ep_len, const double* returns, int64_t n_games, int64_t ptr, int only_solved,
                     int64_t* row_base, int64_t* total_out, void* stream);
/* organise_transitions (Muzero.py:276-323) written as Buffer.add (buffer.py:47-83) into a replay ring
 * of `capacity` rows with buffer.py's arrays (:29-39): states f32[3N], rwds f32[unroll], actions
 * i64[unroll], pi f32[unroll][6], returns f32[unroll], priority f32.  Step t of game g lands in row
 * (row_base[g] + t) % capacity; beyond the episode end the padding is reward 0, return 0, the uniform
 * policy and absorbing_action[g] (the reference draws ONE np.random.randint per episode, :300-303).
 * ep_exp (nullable, uint8 [t_max][n_games]): the play-policy exponent clamp(1/T, 1, 5) that was in force when each move was
 * PLAYED (written by hmz_selfplay_move) — the reference stores the pi_prob run_mcts returned at move time (Muzero.py:179-183),
 * so an episode that spans a change of the temperature schedule keeps each move's own exponent; NULL: `temperature` for all.
 * Rows with row_base[g] + t < first_row are skipped: when one call adds more rows than the ring holds, the
 * reference's one-episode-at-a-time Buffer.add leaves only the LAST `capacity` rows, so the caller passes
 * first_row = ptr + max(0, total - capacity) (0 otherwise). */
int hmz_episode_unroll(const uint32_t* ep_state, const uint8_t* ep_action, const uint8_t* ep_flags, const uint16_t* ep_visits,
                       const double* returns, const float* priority, const int32_t* ep_len, const int64_t* row_base,
                       const uint8_t* absorbing_action, const uint8_t* ep_exp, int64_t n_games, int t_max, int n_disks, int unroll,
                       double temperature, int64_t capacity, int64_t first_row, float* buf_states, float* buf_rwds, int64_t* buf_actions, float* buf_pi,
                       float* buf_returns, float* buf_priority, void* stream);

/* ------------------------------------------------------------------ acting evaluation ------
 * acting_ablations.get_results (acting_experiments/acting_ablations.py:72-128) for parallel episodes.
 * hmz_eval_track, after the env step of move `move_index`: steps[g] <- move_index + 1 when game g's
 * FIRST episode finishes (0 while it runs), illegal_moves[g] counts its illegal moves
 * (illegal_move_rate_comparison.py:27-50).  hmz_eval_errors: errors[g] = steps[g] - min_moves[g]
 * (the hanoi_solver distance of the start state, :96-123), -1 for unfinished games. */
int hmz_eval_track(const uint8_t* flags, int move_index, int64_t n_games, int32_t* steps, int32_t* illegal_moves, void* stream);
int hmz_eval_errors(const int32_t* steps, const uint32_t* min_moves, int64_t n_games, int32_t* errors, void* stream);

/* ------------------------------------------------------------------ learner ----------------
 * Muzero._update (Muzero.py:209-274) + MuZeroNet.update (networks.py:118-122; Adam, networks.py:69) for one batch:
 * the unrolled forward pass, the losses (squared error on the transformed value / reward, cross entropy on the
 * policy, per-sample importance weights, mean, gradient x 1/unroll), the 0.5 gradient hook on the dynamics
 * latents (:235), the backward pass and the Adam step, all float32.
 *   params / grads / adam_m / adam_v: hmz_learner_param_count(n_disks) floats each — the 20 tensors of
 *       MuZeroNet.state_dict() concatenated in state_dict order, each in torch's [out][in] layout
 *   states f32 [batch][3N], rwds / returns f32 [batch][unroll], actions i64 [batch][unroll],
 *   pi_probs f32 [batch][unroll][6], priority_w f32 [batch] or NULL (uniform replay)
 *   step_index: 1 for the first update (Adam bias correction)
 *   new_priorities (nullable) f32 [batch] = |value prediction - return| of unroll step 0 (:253-258)
 *   losses_out f32 [3] (device) = means of the value, reward and policy losses (:269-273)
 *   apply_update == 0: gradients only (grads is an output either way). */
int64_t hmz_learner_param_count(int n_disks);
int64_t hmz_learner_workspace_bytes(int n_disks, int batch, int unroll);
int hmz_learner_step(float* params, float* grads, float* adam_m, float* adam_v, void* workspace, int n_disks, int batch, int unroll,
                     const float* states, const float* rwds, const int64_t* actions, const float* pi_probs, const float* returns,
                     const float* priority_w, double lr, double beta1, double beta2, double eps, int64_t step_index,
                     float* new_priorities, float* losses_out, int apply_update, void* stream);

/* ------------------------------------------------------------------ replay sampling ---------
 * ReplayRing.priority_sample (buffer.py:96) with priority exponent 1, bit-exact with NumPy given the same uniforms:
 *   s = np.sum(q) (float32, NumPy's pairwise tree); x = q / s (float32); np.random.choice(num, batch, p=x), i.e. NumPy's
 *   checks on p = float64(x), cdf = cumsum(p) (float64, left to right, evaluated exactly in parallel), cdf /= cdf[-1],
 *   indices = searchsorted(cdf, uniforms, side="right"); weights = (float32(1 / size) / x[indices]) ** importance_exponent,
 *   weights /= max(weights).
 *   priorities f32 [num] (the filled rows of the ring), uniforms f64 [batch] (np.random.random_sample(batch), the only
 *   draw choice makes), workspace of hmz_replay_sample_workspace_bytes(num) bytes, indices i64 [batch], weights f32 [batch].
 *   *status (device int32) ORs in one HMZ_REPLAY_* bit per error NumPy would raise and is never cleared here, so one
 *   read covers many calls.  The sum check compares the cumulative sum's last value instead of Kahan's sum with the
 *   threshold (they differ by at most num * 2^-53).  importance_exponent 0, 0.5, 1, 2 and -1 are exact (NumPy's fast
 *   paths); others use CUDA's powf.  priority_exponent != 1: HMZ_ERR_UNSUPPORTED; num < 1, size < num, batch < 1:
 *   HMZ_ERR_INVALID; num > 2^27: HMZ_ERR_UNSUPPORTED.
 * hmz_replay_set_priorities: update_priorities (buffer.py:130): if every new priority is finite and one is > 0,
 *   priorities[indices[j]] = new_priorities[j] with the last occurrence of a repeated index winning (NumPy's fancy
 *   assignment); otherwise nothing is written and *status ORs in HMZ_REPLAY_PRIORITY.  Indices outside [0, size) are
 *   skipped. */
#define HMZ_REPLAY_NAN 1u      /* ValueError("probabilities contain NaN")           */
#define HMZ_REPLAY_NEGATIVE 2u /* ValueError("probabilities are not non-negative")  */
#define HMZ_REPLAY_SUM 4u      /* ValueError("probabilities do not sum to 1")       */
#define HMZ_REPLAY_PRIORITY 8u /* AssertionError("Priorities must be finite and positive.") */
int64_t hmz_replay_sample_workspace_bytes(int64_t num);
int hmz_replay_sample(const float* priorities, int64_t num, int64_t size, double priority_exponent, const double* uniforms,
                      int64_t batch, double importance_exponent, void* workspace, int64_t* indices, float* weights, int32_t* status,
                      void* stream);
int hmz_replay_set_priorities(float* priorities, int64_t size, const int64_t* indices, const float* new_priorities, int64_t batch,
                              int32_t* status, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* HMZ_H */
