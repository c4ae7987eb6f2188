// Self-play glue: on-device Dirichlet / uniform draws (throughput mode) and the per-move sequence of
// Muzero._play_game (Muzero.py:153-207 of the reference) around the search — two fused kernels per move:
//   selfplay_begin   the Dirichlet draw + mix (MCTS/mcts.py:132-152), the root record (MCTS/mcts.py:52-69) and the
//                    sampling uniform of the move
//   selfplay_finish  root visit histogram -> play policy -> sampled action (MCTS/mcts.py:112-126), the move's record
//                    (Muzero.py:179-183) in its 32-byte wire form and in the episode store, TowersOfHanoi.step
//                    (env/hanoi.py:47-84) with auto-reset, episode bookkeeping
// Random streams are Philox4x32-10 keyed by (seed, GLOBAL game id, move index): results do not depend on how the
// games are sharded over GPUs (SURVEY.md §8e).
#include "hmz_env.cuh"
#include "hmz_tree.cuh"

namespace hmz {

static_assert(sizeof(hmz_move_record_t) == 32, "wire record (include/hmz.h) must be 32 bytes");

struct PhiloxStream {  // sequential 32-bit draws from one (key, item) Philox stream
  uint32_t c0, c1, c2, c3, k0, k1;
  Philox4 buf;
  int have;
  __device__ PhiloxStream(uint64_t seed, uint64_t item, uint64_t counter)
      : c0((uint32_t)item), c1((uint32_t)(item >> 32)), c2((uint32_t)counter), c3((uint32_t)(counter >> 32) << 8),
        k0((uint32_t)seed), k1((uint32_t)(seed >> 32)), have(0) {}
  __device__ uint32_t next() {
    if (have == 0) {
      buf = philox4x32_10(c0, c1, c2, c3, k0, k1);
      ++c3;  // low 8 bits of c3: up to 256 blocks per (item, counter)
      have = 4;
    }
    --have;
    return have == 3 ? buf.x : (have == 2 ? buf.y : (have == 1 ? buf.z : buf.w));
  }
  __device__ double uniform() {  // (0, 1): 53 random bits, never exactly 0
    const uint64_t hi = next(), lo = next();
    return ((double)(((hi << 32) | lo) >> 11) + 0.5) * (1.0 / 9007199254740992.0);
  }
  __device__ double normal() {  // Box-Muller
    const double u1 = uniform(), u2 = uniform();
    return sqrt(-2.0 * log(u1)) * cospi(2.0 * u2);
  }
  // Marsaglia & Tsang (2000); for alpha < 1: gamma(alpha) = gamma(alpha + 1) * U^(1/alpha)
  __device__ double gamma(double alpha) {
    const double a = alpha < 1.0 ? alpha + 1.0 : alpha;
    const double d = a - 1.0 / 3.0, c = 1.0 / sqrt(9.0 * d);
    double out;
    for (;;) {
      double x = normal(), t = 1.0 + c * x;
      if (t <= 0.0) continue;
      t = t * t * t;
      const double u = uniform();
      if (log(u) < 0.5 * x * x + d - d * t + d * log(t)) {
        out = d * t;
        break;
      }
    }
    if (alpha < 1.0) out *= pow(uniform(), 1.0 / alpha);
    return out;
  }
};

// np.random.dirichlet(alpha * ones(6)) (MCTS/mcts.py:148-149) for global item `item`: six gamma draws, normalised.
// Every action draws from its OWN Philox stream (the key carries the action), so the six draws can be made by six
// lanes at once (selfplay_begin) or one after another (rng_dirichlet) with identical results.
__device__ __forceinline__ double dirichlet_gamma(uint64_t seed, uint64_t item, uint64_t counter, double alpha, int a) {
  PhiloxStream rng(seed ^ 0x4449524943484C45ull ^ ((uint64_t)(a + 1) << 56), item, counter);
  return rng.gamma(alpha);
}
// the six gammas -> the Dirichlet draw (left-to-right sum, as both callers must round identically)
__device__ __forceinline__ void dirichlet_normalise(uint64_t seed, uint64_t item, uint64_t counter, double (&g)[6]) {
  double sum = 0.0;
#pragma unroll
  for (int a = 0; a < 6; ++a) sum += g[a];
  if (!(sum > 0.0)) {  // all six gammas underflowed (alpha tiny): fall back to one-hot on a random action
    PhiloxStream rng(seed ^ 0x4449524943484C45ull ^ (7ull << 56), item, counter);
    const int pick = (int)(rng.uniform() * 6.0);
#pragma unroll
    for (int a = 0; a < 6; ++a) g[a] = (a == pick) ? 1.0 : 0.0;
    sum = 1.0;
  }
#pragma unroll
  for (int a = 0; a < 6; ++a) g[a] = g[a] / sum;
}
__device__ __forceinline__ void dirichlet6(uint64_t seed, uint64_t item, uint64_t counter, double alpha, double (&g)[6]) {
#pragma unroll 1
  for (int a = 0; a < 6; ++a) g[a] = dirichlet_gamma(seed, item, counter, alpha, a);
  dirichlet_normalise(seed, item, counter, g);
}

// One uniform double in [0, 1) for global item `item` (the draw of np.random.choice, MCTS/mcts.py:120).
__device__ __forceinline__ double uniform01(uint64_t seed, uint64_t item, uint64_t counter) {
  const Philox4 r = philox4x32_10((uint32_t)item, (uint32_t)(item >> 32), (uint32_t)counter, (uint32_t)(counter >> 32),
                                  (uint32_t)seed ^ 0x554E4946u, (uint32_t)(seed >> 32));
  return (double)((((uint64_t)r.x << 32) | r.y) >> 11) * (1.0 / 9007199254740992.0);
}

__global__ void __launch_bounds__(256) rng_dirichlet(double* __restrict__ out, int64_t n, double alpha, uint64_t seed,
                                                    uint64_t counter, uint64_t item_offset) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    double g[6];
    dirichlet6(seed, item_offset + (uint64_t)i, counter, alpha, g);
#pragma unroll
    for (int a = 0; a < 6; ++a) out[i * 6 + a] = g[a];
  }
}

__global__ void __launch_bounds__(256) rng_uniform(double* __restrict__ out, int64_t n, uint64_t seed, uint64_t counter,
                                                  uint64_t item_offset) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    out[i] = uniform01(seed, item_offset + (uint64_t)i, counter);
}

__global__ void __launch_bounds__(256) rng_uniform_keyed(double* __restrict__ out, int64_t n, uint64_t seed,
                                                        const uint64_t* __restrict__ counter_hi, uint64_t counter_lo,
                                                        const uint64_t* __restrict__ item) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    out[i] = uniform01(seed, item[i], counter_hi[i] | counter_lo);
}

// Tests: raw Philox4x32-10 blocks (known-answer vectors of Salmon et al. 2011, Random123 kat_vectors).
__global__ void philox_blocks(const uint32_t* __restrict__ ctr_key, uint32_t* __restrict__ out, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t* x = ctr_key + 6 * i;
  const Philox4 r = philox4x32_10(x[0], x[1], x[2], x[3], x[4], x[5]);
  out[4 * i] = r.x;
  out[4 * i + 1] = r.y;
  out[4 * i + 2] = r.z;
  out[4 * i + 3] = r.w;
}

// Start of a move for every game: prior = p0, or add_dirichlet_noise (MCTS/mcts.py:148-150) with the draw made here;
// root_node.expand(prior, h, 0.0) (MCTS/mcts.py:52-69): record 0 <- priors, root.W <- 0; the move's sampling uniform.
// Bit-identical to hmz_rng_dirichlet + hmz_rng_uniform + hmz_search_begin_p0 issued one after another.
// EIGHT lanes per game: lanes 0..5 draw the six gammas in parallel (the rejection sampler in float64 is the whole cost
// of this kernel), every lane then rebuilds the full draw from six shuffles and lanes 0 / 1 write the record halves.
__global__ void __launch_bounds__(256) selfplay_begin(hmz_search_t s, const float* __restrict__ p0, double* __restrict__ noise_out,
                                                     double* __restrict__ uniform_out, double alpha, float one_minus_eps, double eps,
                                                     int use_noise, uint64_t seed, uint64_t counter, uint64_t game_offset) {
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  const int a8 = (int)(t & 7);
  const bool valid = (t >> 3) < s.n_searches;  // whole 8-lane groups are valid or not: the shuffles below stay convergent
  const int64_t b = valid ? (t >> 3) : s.n_searches - 1;
  const uint64_t game = game_offset + (uint64_t)b;
  double mine = 0.0;
  if (use_noise && a8 < 6) mine = dirichlet_gamma(seed, game, counter, alpha, a8);
  double g[6];
#pragma unroll
  for (int a = 0; a < 6; ++a) g[a] = __shfl_sync(0xffffffffu, mine, (threadIdx.x & 24) | a);
  if (use_noise) dirichlet_normalise(seed, game, counter, g);
  if (!valid) return;
  float pr[6];
#pragma unroll
  for (int a = 0; a < 6; ++a) {
    const float q = p0[b * 6 + a];
    double p = (double)q;
    if (use_noise) p = __dadd_rn((double)__fmul_rn(one_minus_eps, q), __dmul_rn(eps, g[a]));  // f32 product, f64 sum
    pr[a] = (float)p;
    if (a == a8) {
      s.root_prior[b * 6 + a] = p;
      if (use_noise && noise_out) noise_out[b * 6 + a] = g[a];
    }
  }
  hmz_node_t* rec = &s.nodes[b * s.n_records];
  if (a8 < 2) write_fresh_half(rec, a8, pr, 0, 0);
  if (a8 == 6) s.root_W[b] = 0.0;
  if (a8 == 7) uniform_out[b] = uniform01(seed, game, counter);
}

// The episode store (include/hmz.h): [t_max][n_games] struct-of-arrays, slot = the game's own step counter.
struct EpisodeStore {
  uint32_t* state;
  uint8_t* action;
  uint8_t* flags;
  uint16_t* visits;
  double* root_q;
  int32_t* cur_slot;
  int32_t* len;
  uint8_t* exp;  // nullable
  int t_max;
};

// The episode-store writes of game b's move (hmz_episode_record + hmz_episode_close in one): slot = the counter bits of the
// env word before the move, clamped to t_max - 1.  The store's two writers, selfplay_finish (from the move itself) and
// episode_ingest (from its gathered wire record), both go through here so that they cannot drift apart.
__device__ __forceinline__ void episode_store_move(const EpisodeStore& e, int64_t n, int64_t b, int n_disks, uint32_t w, int action,
                                                   const int (&visits)[6], double q, uint32_t flags, int exponent) {
  int t = (int)(w >> (2 * n_disks));
  if (t >= e.t_max) t = e.t_max - 1;
  const int64_t at = (int64_t)t * n + b;
  e.state[at] = w;
  e.action[at] = (uint8_t)action;
  e.root_q[at] = q;
#pragma unroll
  for (int k = 0; k < 6; ++k) e.visits[at * 6 + k] = (uint16_t)visits[k];
  e.cur_slot[b] = t;
  e.flags[at] = (uint8_t)flags;
  e.len[b] = (flags & HMZ_FLAG_DONE) ? t + 1 : 0;
  if (e.exp) e.exp[at] = (uint8_t)exponent;
}

struct FinishArgs {
  hmz_search_t s;
  EnvCfg env;
  const double* uniform;
  const double* pow_table;
  uint32_t* words;
  hmz_move_record_t* records;
  int32_t* visits;
  double* root_q;
  int32_t* action;
  EpisodeStore ep;  // ep.state == nullptr: no episode store
  double temperature;
  uint64_t game_offset;
  int n_sims, n_disks, exponent;
};

// End of a move for every game, one thread each: MCTS/mcts.py:112-126 (root_policy_eval), the move's record, the env step.
__global__ void __launch_bounds__(256) selfplay_finish(FinishArgs a) {
  const int64_t n = a.s.n_searches;
  for (int64_t b = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; b < n; b += (int64_t)gridDim.x * blockDim.x) {
    const RootPolicy rp = root_policy_eval(a.s.nodes + b * a.s.n_records, a.temperature, 0, a.uniform[b], a.pow_table, a.n_sims + 1);
    const double q = a.n_sims > 0 ? __ddiv_rn(a.s.root_W[b], (double)a.n_sims) : 0.0;  // Node.Q (node.py:125-131)
    const uint32_t w = a.words[b];
    const StepOut o = step_word(w, (uint32_t)rp.action, a.env);
    a.words[b] = o.word;
    if (a.visits) {
#pragma unroll
      for (int k = 0; k < 6; ++k) a.visits[b * 6 + k] = rp.n[k];
    }
    if (a.root_q) a.root_q[b] = q;
    if (a.action) a.action[b] = rp.action;
    if (a.records) {  // 32 bytes as two 128-bit stores
      const uint64_t game = a.game_offset + (uint64_t)b;
      uint4* dst = reinterpret_cast<uint4*>(a.records + b);
      dst[0] = make_uint4((uint32_t)__double2loint(q), (uint32_t)__double2hiint(q), w, __float_as_uint(o.reward));
      dst[1] = make_uint4((uint32_t)rp.n[0] | ((uint32_t)rp.n[1] << 16), (uint32_t)rp.n[2] | ((uint32_t)rp.n[3] << 16),
                          (uint32_t)rp.n[4] | ((uint32_t)rp.n[5] << 16),
                          (uint32_t)rp.action | (o.flags << 8) | ((uint32_t)(game & 0xFFFFu) << 16));
    }
    if (a.ep.state)  // episode store: slot = the game's own step counter before the move
      episode_store_move(a.ep, n, b, a.n_disks, w, rp.action, rp.n, q, o.flags, a.exponent);
  }
}

// Gathered move records -> the episode store, one thread per record: the store writes selfplay_finish makes, read back from
// the move's 32-byte wire form (two 128-bit loads).  Record b must be global game game_offset + b; one whose game_lo says
// otherwise writes nothing and is counted in *mismatch.
__global__ void __launch_bounds__(256) episode_ingest(const hmz_move_record_t* __restrict__ records, int64_t n, uint64_t game_offset,
                                                     int n_disks, EpisodeStore ep, int exponent, int32_t* __restrict__ mismatch) {
  const int64_t b = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (b >= n) return;
  const uint4* src = reinterpret_cast<const uint4*>(records + b);
  const uint4 r0 = __ldcs(src), r1 = __ldcs(src + 1);  // read once: streaming loads
  if ((r1.w >> 16) != (uint32_t)((game_offset + (uint64_t)b) & 0xFFFFu)) {
    atomicAdd(mismatch, 1);
    return;
  }
  const int visits[6] = {(int)(r1.x & 0xFFFFu), (int)(r1.x >> 16), (int)(r1.y & 0xFFFFu),
                         (int)(r1.y >> 16),     (int)(r1.z & 0xFFFFu), (int)(r1.z >> 16)};
  episode_store_move(ep, n, b, n_disks, r0.z, (int)(r1.w & 0xFFu), visits, __hiloint2double((int)r0.y, (int)r0.x),
                     (r1.w >> 8) & 0xFFu, exponent);
}

// clamp(1/T, 1, 5), MCTS/mcts.py:170-172 (1 for T == 0: raw counts); the episode store keeps integer exponents only
static int play_policy_exponent(const char* who, double temperature, bool store_exp, int* out) {
  double ex = 1.0;
  if (temperature > 0.0) ex = 1.0 / temperature < 1.0 ? 1.0 : (1.0 / temperature > 5.0 ? 5.0 : 1.0 / temperature);
  *out = (int)ex;
  if (store_exp && (double)*out != ex)
    return fail(HMZ_ERR_UNSUPPORTED, "%s: the episode store keeps integer play-policy exponents; temperature %g gives %g", who, temperature, ex);
  return HMZ_OK;
}

}  // namespace hmz

using namespace hmz;

extern "C" {

int hmz_rng_dirichlet(double* out, int64_t n, double alpha, uint64_t seed, uint64_t counter, uint64_t item_offset, void* stream) {
  ProfScope prof_scope(HMZ_PROF_OTHER, stream);
  if (n == 0) return HMZ_OK;
  if (!out || n < 0 || !(alpha > 0.0)) return fail(HMZ_ERR_INVALID, "hmz_rng_dirichlet: bad arguments");
  rng_dirichlet<<<grid_for(n, 256, 4), 256, 0, (cudaStream_t)stream>>>(out, n, alpha, seed, counter, item_offset);
  return check_launch("rng_dirichlet");
}

int hmz_rng_uniform(double* out, int64_t n, uint64_t seed, uint64_t counter, uint64_t item_offset, void* stream) {
  ProfScope prof_scope(HMZ_PROF_OTHER, stream);
  if (n == 0) return HMZ_OK;
  if (!out || n < 0) return fail(HMZ_ERR_INVALID, "hmz_rng_uniform: bad arguments");
  rng_uniform<<<grid_for(n, 256, 8), 256, 0, (cudaStream_t)stream>>>(out, n, seed, counter, item_offset);
  return check_launch("rng_uniform");
}

int hmz_rng_uniform_keyed(double* out, int64_t n, uint64_t seed, const uint64_t* counter_hi, uint64_t counter_lo,
                          const uint64_t* item, void* stream) {
  ProfScope prof_scope(HMZ_PROF_OTHER, stream);
  if (n == 0) return HMZ_OK;
  if (!out || !counter_hi || !item || n < 0) return fail(HMZ_ERR_INVALID, "hmz_rng_uniform_keyed: bad arguments");
  rng_uniform_keyed<<<grid_for(n, 256, 8), 256, 0, (cudaStream_t)stream>>>(out, n, seed, counter_hi, counter_lo, item);
  return check_launch("rng_uniform_keyed");
}

int hmz_debug_philox(const uint32_t* counters_keys, uint32_t* out, int n_blocks, void* stream) {
  if (n_blocks <= 0) return HMZ_OK;
  if (!counters_keys || !out) return fail(HMZ_ERR_INVALID, "hmz_debug_philox: null pointer");
  philox_blocks<<<(n_blocks + 127) / 128, 128, 0, (cudaStream_t)stream>>>(counters_keys, out, n_blocks);
  return check_launch("philox_blocks");
}

// One move of every game (Muzero._play_game loop body, Muzero.py:165-186): root inference -> Dirichlet mix + root
// record -> n_simulations fused simulations -> root policy + sampled action + move record + env step.
// Four launches around the search: no host synchronisation, everything on `stream`.
int hmz_selfplay_move(const hmz_selfplay_t* sp, uint64_t move_index, void* stream) {
  if (!sp) return fail(HMZ_ERR_INVALID, "hmz_selfplay_move: null descriptor");
  const hmz_search_t* s = &sp->search;
  const int64_t B = s->n_searches;
  if (B == 0) return HMZ_OK;
  if (!sp->weights || !sp->words || !sp->p0 || !sp->v0 || !sp->uniform || !sp->ucb_table || B < 0)
    return fail(HMZ_ERR_INVALID, "hmz_selfplay_move: null buffer in descriptor");
  const bool use_noise = sp->dirichlet_alpha > 0.0 && sp->exploration_eps > 0.0;
  if (s->root_prior_is_f64 != (use_noise ? 1 : 0))
    return fail(HMZ_ERR_INVALID, "hmz_selfplay_move: search.root_prior_is_f64 must be %d", use_noise ? 1 : 0);
  if (!(sp->temperature >= 0.0 && sp->temperature <= 1.0))  // MCTS/mcts.py:163-166
    return fail(HMZ_ERR_INVALID, "Expect `temperature` to be in the range [0.0, 1.0], got %g", sp->temperature);
  const bool ep = sp->ep_state != nullptr;
  if (ep && (!sp->ep_action || !sp->ep_flags || !sp->ep_visits || !sp->ep_root_q || !sp->ep_cur_slot || !sp->ep_len || sp->ep_t_max < 1))
    return fail(HMZ_ERR_INVALID, "hmz_selfplay_move: incomplete episode store");
  if (sp->records && (reinterpret_cast<uintptr_t>(sp->records) & 15u) != 0)
    return fail(HMZ_ERR_INVALID, "hmz_selfplay_move: records must be 16-byte aligned");
  FinishArgs fa;
  if (int rc = make_env_cfg(fa.env, sp->n_disks, sp->max_steps, sp->goal_peg, 1, sp->reset_word)) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  if (int rc = hmz_net_initial(sp->weights, sp->mode, sp->n_disks, sp->words, nullptr, s->latents, s->n_records, s->latent_dtype,
                               sp->p0, sp->v0, B, stream))
    return rc;
  {
    ProfScope prof_scope(HMZ_PROF_OTHER, stream);
    if (int rc = check_search(s, "hmz_selfplay_move")) return rc;
    selfplay_begin<<<(unsigned)((B * 8 + 255) / 256), 256, 0, st>>>(*s, sp->p0, sp->noise, sp->uniform, sp->dirichlet_alpha,
                                                                (float)(1.0 - sp->exploration_eps), sp->exploration_eps,
                                                                use_noise ? 1 : 0, sp->seed, move_index, sp->game_offset);
    if (int rc = check_launch("selfplay_begin")) return rc;
  }
  if (int rc = hmz_search_run(s, sp->weights, sp->mode, sp->n_simulations, sp->ucb_table, sp->discount, stream)) return rc;
  ProfScope prof_scope(HMZ_PROF_ROOT_POLICY, stream);
  fa.s = *s;
  fa.uniform = sp->uniform;
  fa.pow_table = sp->pow_table;
  fa.words = sp->words;
  fa.records = sp->records;
  fa.visits = sp->visits;
  fa.root_q = sp->root_q;
  fa.action = sp->action;
  fa.ep = EpisodeStore{sp->ep_state, sp->ep_action, sp->ep_flags, sp->ep_visits, sp->ep_root_q, sp->ep_cur_slot, sp->ep_len,
                       sp->ep_exp, sp->ep_t_max};
  if (int rc = play_policy_exponent("hmz_selfplay_move", sp->temperature, sp->ep_exp != nullptr, &fa.exponent)) return rc;
  fa.temperature = sp->temperature;
  fa.game_offset = sp->game_offset;
  fa.n_sims = sp->n_simulations;
  fa.n_disks = sp->n_disks;
  selfplay_finish<<<grid_for(B, 256, 4), 256, 0, st>>>(fa);
  return check_launch("selfplay_finish");
}

int hmz_episode_ingest(const hmz_move_record_t* records, int64_t n_games, uint64_t game_offset, int n_disks, int t_max,
                       double temperature, uint32_t* ep_state, uint8_t* ep_action, uint8_t* ep_flags, uint16_t* ep_visits,
                       double* ep_root_q, int32_t* cur_slot, int32_t* ep_len, uint8_t* ep_exp, int32_t* mismatch, void* stream) {
  if (!records || !ep_state || !ep_action || !ep_flags || !ep_visits || !ep_root_q || !cur_slot || !ep_len || !mismatch)
    return fail(HMZ_ERR_INVALID, "hmz_episode_ingest: null pointer");
  if (n_games < 0 || t_max < 1 || n_disks < 1 || n_disks > HMZ_MAX_DISKS)
    return fail(HMZ_ERR_INVALID, "hmz_episode_ingest: bad sizes (n_games %lld, t_max %d, n_disks %d)", (long long)n_games, t_max, n_disks);
  if ((reinterpret_cast<uintptr_t>(records) & 15u) != 0) return fail(HMZ_ERR_INVALID, "hmz_episode_ingest: records must be 16-byte aligned");
  if (!(temperature >= 0.0 && temperature <= 1.0))  // MCTS/mcts.py:163-166
    return fail(HMZ_ERR_INVALID, "Expect `temperature` to be in the range [0.0, 1.0], got %g", temperature);
  int exponent;
  if (int rc = play_policy_exponent("hmz_episode_ingest", temperature, ep_exp != nullptr, &exponent)) return rc;
  if (n_games == 0) return HMZ_OK;
  ProfScope prof_scope(HMZ_PROF_OTHER, stream);
  const EpisodeStore ep{ep_state, ep_action, ep_flags, ep_visits, ep_root_q, cur_slot, ep_len, ep_exp, t_max};
  episode_ingest<<<(unsigned)((n_games + 255) / 256), 256, 0, (cudaStream_t)stream>>>(records, n_games, game_offset, n_disks, ep,
                                                                                     exponent, mismatch);
  return check_launch("episode_ingest");
}

}  // extern "C"
