// Episode post-processing on the device (SURVEY.md §8f rows 1-2): the tail of Muzero._play_game
// (reference Muzero.py:189-205) — n-step TD returns (utils.py:28-72), priorities |return - rootQ|
// (Muzero.py:197-200), organise_transitions (Muzero.py:276-323) — written straight into the rows of a
// GPU-resident replay ring with buffer.py's layout (:29-39) and wrap-around (:47-62).
//
// Episode store: struct-of-arrays [t_max][n_games] indexed by the GAME'S OWN step counter (the counter
// bits of its env word), so slots [0, ep_len[g]) of game g hold its current episode:
//   ep_state u32 (env word before the move), ep_action u8, ep_flags u8 (HMZ_FLAG_* of the move: the
//   reward is a function of them), ep_visits u16[6], ep_root_q f64.
//
// Arithmetic contract (bit-exact vs the reference run under CPython >= 3.12):
//   reward           python numbers 0, 100, -100/1000 selected by the flags (env/hanoi.py:62,66,72)
//   discount ** i    host libm values supplied as a table (like the pUCT table: no device pow())
//   sum([...])       CPython's float sum: first add exact, then Neumaier-compensated (bltinmodule.c)
//   everything float64 with explicit round-to-nearest ops (no FMA contraction), cast to float32 where
//   NumPy does (priority operands, replay rows).
#include <cstdlib>

#include "hmz_common.cuh"

namespace hmz {

__device__ __forceinline__ double reward_of(uint32_t flags) {
  if (flags & HMZ_FLAG_GOAL) return 100.0;
  if (flags & HMZ_FLAG_ILLEGAL) return -100.0 / 1000.0;
  return 0.0;
}

// One move of every game into its episode slot (Muzero.py:179-183); remembers the slot for episode_close.
__global__ void __launch_bounds__(256) episode_record(const uint32_t* __restrict__ words, const int32_t* __restrict__ action,
                                                     const int32_t* __restrict__ visits, const double* __restrict__ root_q,
                                                     int n_disks, int t_max, int64_t n, uint32_t* __restrict__ ep_state,
                                                     uint8_t* __restrict__ ep_action, uint16_t* __restrict__ ep_visits,
                                                     double* __restrict__ ep_root_q, int32_t* __restrict__ cur_slot,
                                                     uint8_t* __restrict__ action_u8) {
  for (int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; g < n; g += (int64_t)gridDim.x * blockDim.x) {
    const uint32_t w = words[g];
    int t = (int)(w >> (2 * n_disks));
    if (t >= t_max) t = t_max - 1;  // cannot happen when t_max >= max_steps; keeps the store in bounds
    const int64_t at = (int64_t)t * n + g;
    const uint8_t a = (uint8_t)action[g];
    ep_state[at] = w;
    ep_action[at] = a;
    ep_root_q[at] = root_q[g];
#pragma unroll
    for (int k = 0; k < 6; ++k) ep_visits[at * 6 + k] = (uint16_t)visits[g * 6 + k];
    cur_slot[g] = t;
    if (action_u8) action_u8[g] = a;
  }
}

// After the env step: the move's flags join the slot; a finished game publishes its episode length.
__global__ void __launch_bounds__(256) episode_close(const uint8_t* __restrict__ flags, const int32_t* __restrict__ cur_slot,
                                                    int64_t n, uint8_t* __restrict__ ep_flags, int32_t* __restrict__ ep_len) {
  for (int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; g < n; g += (int64_t)gridDim.x * blockDim.x) {
    const int t = cur_slot[g];
    const uint8_t f = flags[g];
    ep_flags[(int64_t)t * n + g] = f;
    ep_len[g] = (f & HMZ_FLAG_DONE) ? t + 1 : 0;  // 0 = episode still running
  }
}

// compute_n_step_returns (utils.py:28-72) + priorities (Muzero.py:197-200), one thread per (step, game).
__global__ void __launch_bounds__(256) episode_returns(const uint8_t* __restrict__ ep_flags, const double* __restrict__ ep_root_q,
                                                      const int32_t* __restrict__ ep_len, int64_t n, int t_max,
                                                      const double* __restrict__ discount_pow, int n_step,
                                                      double* __restrict__ returns, float* __restrict__ priority) {
  const int64_t total = (int64_t)t_max * n;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t g = i % n;
    const int t = (int)(i / n), len = ep_len[g];
    if (t >= len) continue;
    // sum([discount**i * r for i, r in enumerate(_rwds[t : t + n_step])]) with CPython's float sum
    double f = 0.0, c = 0.0;
    for (int k = 0; k < n_step; ++k) {
      const double r = (t + k < len) ? reward_of(ep_flags[(int64_t)(t + k) * n + g]) : 0.0;  // padding: int 0
      const double x = __dmul_rn(discount_pow[k], r);
      if (k == 0) {
        f = __dadd_rn(0.0, x);  // int 0 + float
      } else {
        const double s = __dadd_rn(f, x);
        if (fabs(f) >= fabs(x))
          c = __dadd_rn(c, __dadd_rn(__dsub_rn(f, s), x));
        else
          c = __dadd_rn(c, __dadd_rn(__dsub_rn(x, s), f));
        f = s;
      }
    }
    if (c != 0.0 && isfinite(c)) f = __dadd_rn(f, c);
    const double boot = (t + n_step < len) ? ep_root_q[(int64_t)(t + n_step) * n + g] : 0.0;  // padding: int 0
    const double value = __dadd_rn(f, __dmul_rn(discount_pow[n_step], boot));
    returns[i] = value;
    if (priority) priority[i] = fabsf(__fsub_rn((float)value, (float)ep_root_q[i]));
  }
}

// compute_MCreturns (utils.py:75-86, the TD_return = False branch of Muzero._play_game) + priorities: one thread
// per game walks its episode from the end — np.cumsum over the flipped discounted rewards is a sequential
// float64 sum — and divides by the discount of each step.  discount_pow[i] = discount ** i as NumPy's power
// ufunc evaluates it (its vectorised pow differs from libm's in the last bit for some exponents).
__global__ void __launch_bounds__(256) episode_mc_returns(const uint8_t* __restrict__ ep_flags, const double* __restrict__ ep_root_q,
                                                         const int32_t* __restrict__ ep_len, int64_t n, int t_max,
                                                         const double* __restrict__ discount_pow, double* __restrict__ returns,
                                                         float* __restrict__ priority) {
  for (int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; g < n; g += (int64_t)gridDim.x * blockDim.x) {
    const int len = ep_len[g] < t_max ? ep_len[g] : t_max;
    double acc = 0.0;
    for (int t = len - 1; t >= 0; --t) {
      const int64_t at = (int64_t)t * n + g;
      const double d = discount_pow[t];
      const double x = __dmul_rn(d, reward_of(ep_flags[at]));
      acc = (t == len - 1) ? x : __dadd_rn(acc, x);
      const double value = __ddiv_rn(acc, d);
      returns[at] = value;
      if (priority) priority[at] = fabsf(__fsub_rn((float)value, (float)ep_root_q[at]));
    }
  }
}

// Which finished episodes enter the replay ring (training_loop stores an episode only if
// returns[-1, 0] > 0, Muzero.py:98) and where: row_base[g] = ptr + exclusive prefix sum of the stored
// lengths (mod capacity applied by the writer), -1 for games that store nothing.  One block; the batch
// is scanned in chunks of blockDim with a running carry.
__global__ void __launch_bounds__(1024) episode_rows(const int32_t* __restrict__ ep_len, const double* __restrict__ returns,
                                                    int64_t n, int64_t ptr, int only_solved, int64_t* __restrict__ row_base,
                                                    int64_t* __restrict__ total_out) {
  __shared__ int64_t warp_sums[32];
  __shared__ int64_t carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int64_t base = 0; base < n; base += blockDim.x) {
    const int64_t g = base + threadIdx.x;
    int64_t len = 0;
    if (g < n) {
      len = ep_len[g];
      if (len > 0 && only_solved && !(returns[(len - 1) * n + g] > 0.0)) len = 0;
    }
    int64_t x = len;  // inclusive scan inside the warp
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int64_t y = __shfl_up_sync(0xffffffffu, x, d);
      if (lane >= d) x += y;
    }
    if (lane == 31) warp_sums[warp] = x;
    __syncthreads();
    if (warp == 0) {
      int64_t s = lane < (int)(blockDim.x >> 5) ? warp_sums[lane] : 0;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const int64_t y = __shfl_up_sync(0xffffffffu, s, d);
        if (lane >= d) s += y;
      }
      warp_sums[lane] = s;  // inclusive over warps
    }
    __syncthreads();
    const int64_t before = carry + (warp > 0 ? warp_sums[warp - 1] : 0) + (x - len);
    if (g < n) row_base[g] = len > 0 ? ptr + before : -1;
    __syncthreads();
    if (threadIdx.x == 0) carry += warp_sums[(blockDim.x >> 5) - 1];
    __syncthreads();
  }
  if (threadIdx.x == 0) *total_out = carry;
}

// organise_transitions (Muzero.py:276-323) + Buffer.add (buffer.py:47-83): one thread per (step, game)
// writes the replay row of that step.
__global__ void __launch_bounds__(256) episode_unroll(
    const uint32_t* __restrict__ ep_state, const uint8_t* __restrict__ ep_action, const uint8_t* __restrict__ ep_flags,
    const uint16_t* __restrict__ ep_visits, const double* __restrict__ returns, const float* __restrict__ priority,
    const int32_t* __restrict__ ep_len, const int64_t* __restrict__ row_base, const uint8_t* __restrict__ absorbing_action,
    const uint8_t* __restrict__ ep_exp, int64_t n, int t_max, int n_disks, int unroll, int exponent, int64_t capacity, int64_t first_row, float* __restrict__ buf_states,
    float* __restrict__ buf_rwds, int64_t* __restrict__ buf_actions, float* __restrict__ buf_pi, float* __restrict__ buf_returns,
    float* __restrict__ buf_priority) {
  const int64_t total = (int64_t)t_max * n;
  const int d_state = 3 * n_disks;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t g = i % n;
    const int t = (int)(i / n), len = ep_len[g];
    const int64_t rb = row_base[g];
    if (t >= len || rb < 0 || rb + t < first_row) continue;  // rows a later row of this add overwrites are skipped
    const int64_t row = (rb + t) % capacity;  // buffer.py:47-62 wrap-around
    // state: utils.oneHot_encoding (utils.py:9-25) of the env word, float32 (buffer.py:29)
    const uint32_t w = ep_state[i];
    for (int d = 0; d < n_disks; ++d) {
      const uint32_t peg = (w >> (2 * d)) & 3u;
#pragma unroll
      for (int p = 0; p < 3; ++p) buf_states[row * d_state + 3 * d + p] = (peg == (uint32_t)p) ? 1.0f : 0.0f;
    }
    buf_priority[row] = priority[i];
    for (int k = 0; k < unroll; ++k) {
      const int j = t + k;
      const int64_t o = row * unroll + k;
      if (j < len) {
        const int64_t at = (int64_t)j * n + g;
        buf_rwds[o] = (float)reward_of(ep_flags[at]);
        buf_actions[o] = (int64_t)ep_action[at];
        buf_returns[o] = (float)returns[at];
        // generate_play_policy (MCTS/mcts.py:154-176): visits ** exponent / sum, float64, then float32 rows
        double wv[6];
#pragma unroll
        for (int a = 0; a < 6; ++a) {
          const double x = (double)ep_visits[at * 6 + a];
          double y = x;
          const int ex_at = ep_exp ? (int)ep_exp[at] : exponent;  // the exponent in force when the move was played
          for (int e = 1; e < ex_at; ++e) y = __dmul_rn(y, x);
          wv[a] = y;
        }
        double tot = wv[0];  // np.sum of 6 doubles: left to right (NumPy sums arrays shorter than 8 sequentially)
#pragma unroll
        for (int a = 1; a < 6; ++a) tot = __dadd_rn(tot, wv[a]);
#pragma unroll
        for (int a = 0; a < 6; ++a) buf_pi[o * 6 + a] = (float)__ddiv_rn(wv[a], tot);
      } else {  // absorbing padding (Muzero.py:296-307): reward 0, return 0, one random action, uniform policy
        buf_rwds[o] = 0.0f;
        buf_actions[o] = (int64_t)absorbing_action[g];
        buf_returns[o] = 0.0f;
#pragma unroll
        for (int a = 0; a < 6; ++a) buf_pi[o * 6 + a] = (float)(1.0 / 6.0);
      }
    }
  }
}


// Same rows, one WARP per game: the episode's per-step inputs are gathered once into shared memory (the
// [t][game] store makes those reads one sector each), the play policy is evaluated once per step instead of once
// per (row, unroll slot), and every output array is then written with consecutive lanes on consecutive words —
// rows of one episode are consecutive in the ring, so the stores are full 128-byte lines.
struct StepStage {  // 44 bytes per episode step
  float reward, ret, priority;
  uint32_t state;
  float pi[6];
  uint32_t action;
};
__global__ void __launch_bounds__(128) episode_unroll_warp(
    const uint32_t* __restrict__ ep_state, const uint8_t* __restrict__ ep_action, const uint8_t* __restrict__ ep_flags,
    const uint16_t* __restrict__ ep_visits, const double* __restrict__ returns, const float* __restrict__ priority,
    const int32_t* __restrict__ ep_len, const int64_t* __restrict__ row_base, const uint8_t* __restrict__ absorbing_action,
    const uint8_t* __restrict__ ep_exp, int64_t n, int t_max, int n_disks, int unroll, int exponent, int64_t capacity, int64_t first_row, float* __restrict__ buf_states,
    float* __restrict__ buf_rwds, int64_t* __restrict__ buf_actions, float* __restrict__ buf_pi, float* __restrict__ buf_returns,
    float* __restrict__ buf_priority) {
  extern __shared__ StepStage stage_all[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, warps = blockDim.x >> 5;
  StepStage* stage = stage_all + (size_t)warp * t_max;
  const int d_state = 3 * n_disks;
  for (int64_t g = (int64_t)blockIdx.x * warps + warp; g < n; g += (int64_t)gridDim.x * warps) {
    const int len = ep_len[g] < t_max ? ep_len[g] : t_max;
    const int64_t rb = row_base[g];
    if (len <= 0 || rb < 0) continue;  // warp-uniform
    __syncwarp();
    for (int t = lane; t < len; t += 32) {
      const int64_t at = (int64_t)t * n + g;
      StepStage st;
      st.reward = (float)reward_of(ep_flags[at]);
      st.ret = (float)returns[at];
      st.priority = priority[at];
      st.state = ep_state[at];
      st.action = ep_action[at];
      double wv[6];  // generate_play_policy (MCTS/mcts.py:154-176): visits ** exponent / sum, float64, then float32 rows
#pragma unroll
      for (int a = 0; a < 6; ++a) {
        const double x = (double)ep_visits[at * 6 + a];
        double y = x;
        const int ex_at = ep_exp ? (int)ep_exp[at] : exponent;  // the exponent in force when the move was played
        for (int e = 1; e < ex_at; ++e) y = __dmul_rn(y, x);
        wv[a] = y;
      }
      double tot = wv[0];  // np.sum of 6 doubles: left to right (NumPy sums arrays shorter than 8 sequentially)
#pragma unroll
      for (int a = 1; a < 6; ++a) tot = __dadd_rn(tot, wv[a]);
#pragma unroll
      for (int a = 0; a < 6; ++a) st.pi[a] = (float)__ddiv_rn(wv[a], tot);
      stage[t] = st;
    }
    __syncwarp();
    const int64_t absorbing = (int64_t)absorbing_action[g];
    const float uniform = (float)(1.0 / 6.0);
    // states [len][3N]: utils.oneHot_encoding of the env word
    for (int w = lane; w < len * d_state; w += 32) {
      const int t = w / d_state, c = w - t * d_state, d = c / 3;
      if (rb + t < first_row) continue;  // overwritten by a later row of this add (more rows than the ring holds)
      buf_states[((rb + t) % capacity) * d_state + c] = (((stage[t].state >> (2 * d)) & 3u) == (uint32_t)(c - 3 * d)) ? 1.0f : 0.0f;
    }
    for (int t = lane; t < len; t += 32)
      if (rb + t >= first_row) buf_priority[(rb + t) % capacity] = stage[t].priority;
    // [len][unroll] arrays: rewards, returns, actions; beyond the episode end the absorbing padding (Muzero.py:296-307)
    for (int w = lane; w < len * unroll; w += 32) {
      const int t = w / unroll, k = w - t * unroll, j = t + k;
      if (rb + t < first_row) continue;
      const int64_t o = ((rb + t) % capacity) * unroll + k;
      buf_rwds[o] = j < len ? stage[j].reward : 0.0f;
      buf_returns[o] = j < len ? stage[j].ret : 0.0f;
      buf_actions[o] = j < len ? (int64_t)stage[j].action : absorbing;
    }
    for (int w = lane; w < len * unroll * 6; w += 32) {
      const int t = w / (unroll * 6), r = w - t * unroll * 6, k = r / 6, a = r - k * 6, j = t + k;
      if (rb + t < first_row) continue;
      buf_pi[((rb + t) % capacity) * unroll * 6 + r] = j < len ? stage[j].pi[a] : uniform;
    }
  }
}

}  // namespace hmz

using namespace hmz;

extern "C" {

int hmz_episode_record(const uint32_t* words, const int32_t* action, const int32_t* visits, const double* root_q, int n_disks,
                       int t_max, int64_t n_games, uint32_t* ep_state, uint8_t* ep_action, uint16_t* ep_visits,
                       double* ep_root_q, int32_t* cur_slot, uint8_t* action_u8_out, void* stream) {
  ProfScope prof_scope(HMZ_PROF_OTHER, stream);
  if (n_games == 0) return HMZ_OK;
  if (!words || !action || !visits || !root_q || !ep_state || !ep_action || !ep_visits || !ep_root_q || !cur_slot ||
      n_games < 0 || t_max < 1 || n_disks < 1 || n_disks > HMZ_MAX_DISKS)
    return fail(HMZ_ERR_INVALID, "hmz_episode_record: bad arguments");
  episode_record<<<grid_for(n_games, 256, 8), 256, 0, (cudaStream_t)stream>>>(words, action, visits, root_q, n_disks, t_max, n_games,
                                                                              ep_state, ep_action, ep_visits, ep_root_q, cur_slot,
                                                                              action_u8_out);
  return check_launch("episode_record");
}

int hmz_episode_close(const uint8_t* flags, const int32_t* cur_slot, int64_t n_games, uint8_t* ep_flags, int32_t* ep_len,
                      void* stream) {
  ProfScope prof_scope(HMZ_PROF_OTHER, stream);
  if (n_games == 0) return HMZ_OK;
  if (!flags || !cur_slot || !ep_flags || !ep_len || n_games < 0) return fail(HMZ_ERR_INVALID, "hmz_episode_close: bad arguments");
  episode_close<<<grid_for(n_games, 256, 8), 256, 0, (cudaStream_t)stream>>>(flags, cur_slot, n_games, ep_flags, ep_len);
  return check_launch("episode_close");
}

int hmz_episode_returns(const uint8_t* ep_flags, const double* ep_root_q, const int32_t* ep_len, int64_t n_games, int t_max,
                        const double* discount_pow, int n_step, double* returns, float* priority, void* stream) {
  ProfScope prof_scope(HMZ_PROF_OTHER, stream);
  if (n_games == 0) return HMZ_OK;
  if (!ep_flags || !ep_root_q || !ep_len || !discount_pow || !returns || n_games < 0 || t_max < 1 || n_step < 1)
    return fail(HMZ_ERR_INVALID, "hmz_episode_returns: bad arguments (n_step must be > 0, utils.py:44)");
  episode_returns<<<grid_for(n_games * t_max, 256, 8), 256, 0, (cudaStream_t)stream>>>(ep_flags, ep_root_q, ep_len, n_games, t_max,
                                                                                       discount_pow, n_step, returns, priority);
  return check_launch("episode_returns");
}

int hmz_episode_mc_returns(const uint8_t* ep_flags, const double* ep_root_q, const int32_t* ep_len, int64_t n_games, int t_max,
                           const double* discount_pow, double* returns, float* priority, void* stream) {
  ProfScope prof_scope(HMZ_PROF_OTHER, stream);
  if (n_games == 0) return HMZ_OK;
  if (!ep_flags || !ep_len || !discount_pow || !returns || (priority && !ep_root_q) || n_games < 0 || t_max < 1)
    return fail(HMZ_ERR_INVALID, "hmz_episode_mc_returns: bad arguments");
  episode_mc_returns<<<grid_for(n_games, 256, 8), 256, 0, (cudaStream_t)stream>>>(ep_flags, ep_root_q, ep_len, n_games, t_max,
                                                                                  discount_pow, returns, priority);
  return check_launch("episode_mc_returns");
}

int hmz_episode_rows(const int32_t* ep_len, const double* returns, int64_t n_games, int64_t ptr, int only_solved,
                     int64_t* row_base, int64_t* total_out, void* stream) {
  ProfScope prof_scope(HMZ_PROF_OTHER, stream);
  if (!total_out) return fail(HMZ_ERR_INVALID, "hmz_episode_rows: null total_out");
  if (n_games < 0 || (n_games > 0 && (!ep_len || !row_base || (only_solved && !returns))) || ptr < 0)
    return fail(HMZ_ERR_INVALID, "hmz_episode_rows: bad arguments");
  episode_rows<<<1, 1024, 0, (cudaStream_t)stream>>>(ep_len, returns, n_games, ptr, only_solved, row_base, total_out);
  return check_launch("episode_rows");
}

int hmz_episode_unroll(const uint32_t* ep_state, const uint8_t* ep_action, const uint8_t* ep_flags, const uint16_t* ep_visits,
                       const double* returns, const float* priority, const int32_t* ep_len, const int64_t* row_base,
                       const uint8_t* absorbing_action, const uint8_t* ep_exp, int64_t n_games, int t_max, int n_disks, int unroll,
                       double temperature, int64_t capacity, int64_t first_row, float* buf_states, float* buf_rwds, int64_t* buf_actions, float* buf_pi,
                       float* buf_returns, float* buf_priority, void* stream) {
  ProfScope prof_scope(HMZ_PROF_OTHER, stream);
  if (n_games == 0) return HMZ_OK;
  if (!(temperature >= 0.0 && temperature <= 1.0))  // MCTS/mcts.py:163-166
    return fail(HMZ_ERR_INVALID, "Expect `temperature` to be in the range [0.0, 1.0], got %g", temperature);
  if (!ep_state || !ep_action || !ep_flags || !ep_visits || !returns || !priority || !ep_len || !row_base || !absorbing_action ||
      !buf_states || !buf_rwds || !buf_actions || !buf_pi || !buf_returns || !buf_priority || n_games < 0 || t_max < 1 ||
      n_disks < 1 || n_disks > HMZ_MAX_DISKS || unroll < 1 || capacity < 1)
    return fail(HMZ_ERR_INVALID, "hmz_episode_unroll: bad arguments");
  // visits ** max(1, min(5, 1/T)) for T > 0, raw counts for T == 0 (MCTS/mcts.py:168-174); the reference's
  // temperature schedule (utils.py:89-96) only produces the integer exponents 1, 2, 5 (10 clamps to 5).
  double ex = 1.0;
  if (temperature > 0.0) ex = 1.0 / temperature < 1.0 ? 1.0 : (1.0 / temperature > 5.0 ? 5.0 : 1.0 / temperature);
  const int iex = (int)ex;
  if ((double)iex != ex)
    return fail(HMZ_ERR_UNSUPPORTED, "hmz_episode_unroll: temperature %g gives the non-integer exponent %g", temperature, ex);
  const size_t stage_bytes = (size_t)t_max * sizeof(StepStage);
  if (stage_bytes * 4 <= 48 * 1024 && !getenv("HMZ_UNROLL_SCALAR")) {  // warp-per-game form: staging fits the default shared memory
    episode_unroll_warp<<<grid_for(n_games, 4, 8), 128, stage_bytes * 4, (cudaStream_t)stream>>>(
        ep_state, ep_action, ep_flags, ep_visits, returns, priority, ep_len, row_base, absorbing_action, ep_exp, n_games, t_max, n_disks,
        unroll, iex, capacity, first_row, buf_states, buf_rwds, buf_actions, buf_pi, buf_returns, buf_priority);
    return check_launch("episode_unroll_warp");
  }
  episode_unroll<<<grid_for(n_games * t_max, 256, 8), 256, 0, (cudaStream_t)stream>>>(
      ep_state, ep_action, ep_flags, ep_visits, returns, priority, ep_len, row_base, absorbing_action, ep_exp, n_games, t_max, n_disks, unroll,
      iex, capacity, first_row, buf_states, buf_rwds, buf_actions, buf_pi, buf_returns, buf_priority);
  return check_launch("episode_unroll");
}

}  // extern "C"

// ---- acting evaluation (acting_experiments/acting_ablations.py:72-128) --------------------------
// Per game: the length of its FIRST episode (`step` when `done` first turns true, :104-123) and the
// number of illegal moves in it (illegal_move_rate_comparison.py:27-50).  steps[g] == 0 means the
// first episode is still running.
namespace hmz {
__global__ void __launch_bounds__(256) eval_track(const uint8_t* __restrict__ flags, int move_index, int64_t n,
                                                 int32_t* __restrict__ steps, int32_t* __restrict__ illegal_moves) {
  for (int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; g < n; g += (int64_t)gridDim.x * blockDim.x) {
    if (steps[g] != 0) continue;
    const uint8_t f = flags[g];
    if (f & HMZ_FLAG_ILLEGAL) illegal_moves[g] += 1;
    if (f & HMZ_FLAG_DONE) steps[g] = move_index + 1;
  }
}
// errors[g] = steps[g] - hanoi_solver(start state) (acting_ablations.py:96-123); -1 while unfinished
__global__ void __launch_bounds__(256) eval_errors(const int32_t* __restrict__ steps, const uint32_t* __restrict__ min_moves,
                                                  int64_t n, int32_t* __restrict__ errors) {
  for (int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; g < n; g += (int64_t)gridDim.x * blockDim.x)
    errors[g] = steps[g] > 0 ? steps[g] - (int32_t)min_moves[g] : -1;
}
}  // namespace hmz

extern "C" {

int hmz_eval_track(const uint8_t* flags, int move_index, int64_t n_games, int32_t* steps, int32_t* illegal_moves, void* stream) {
  hmz::ProfScope prof_scope(HMZ_PROF_OTHER, stream);
  if (n_games == 0) return HMZ_OK;
  if (!flags || !steps || !illegal_moves || n_games < 0 || move_index < 0)
    return hmz::fail(HMZ_ERR_INVALID, "hmz_eval_track: bad arguments");
  hmz::eval_track<<<hmz::grid_for(n_games, 256, 8), 256, 0, (cudaStream_t)stream>>>(flags, move_index, n_games, steps, illegal_moves);
  return hmz::check_launch("eval_track");
}

int hmz_eval_errors(const int32_t* steps, const uint32_t* min_moves, int64_t n_games, int32_t* errors, void* stream) {
  hmz::ProfScope prof_scope(HMZ_PROF_OTHER, stream);
  if (n_games == 0) return HMZ_OK;
  if (!steps || !min_moves || !errors || n_games < 0) return hmz::fail(HMZ_ERR_INVALID, "hmz_eval_errors: bad arguments");
  hmz::eval_errors<<<hmz::grid_for(n_games, 256, 8), 256, 0, (cudaStream_t)stream>>>(steps, min_moves, n_games, errors);
  return hmz::check_launch("eval_errors");
}

}  // extern "C"
