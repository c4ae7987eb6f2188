// Vectorised Tower-of-Hanoi environment kernels (sm_100a).
//
// Restates env/hanoi.py of the reference (TowersOfHanoi.step :47-84, _move_allowed :123-139,
// _get_moved_state :141-151, reset :86-96, random_reset :98-111), utils.oneHot_encoding
// (utils.py:9-25) and env/hanoi_utils.hanoi_solver (:4-26) on packed 32-bit env words.
//
// All kernels are HBM-streaming integer kernels: one env word per lane, 4 words per thread
// through 128-bit loads/stores, grids sized in whole waves of the SM count.  No tensor cores:
// there is no contraction here.
#include "hmz_env.cuh"

namespace hmz {

// ------------------------------------------------------------------------------ kernels
// One thread owns one vec4 group per grid-stride iteration, so that every load / store instruction of a warp covers one
// contiguous 512-byte (words, rewards) or 128-byte (actions, flags) span.  Measured on the B200 (2^24 envs), with U vec4
// groups per thread and iteration: U = 1 4.19-4.26 TB/s, U = 2 4.0, U = 4 3.9 — more bytes in flight per thread do not
// help (2,048 resident threads per SM already cover the latency-bandwidth product); the unrolled forms have been removed.
template <bool kObs>
__global__ void __launch_bounds__(256) env_step_vec4(uint4* __restrict__ words, const uchar4* __restrict__ actions,
                                                    float4* __restrict__ rewards, uchar4* __restrict__ flags,
                                                    uint4* __restrict__ obs_words, int64_t n_vec, EnvCfg c) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n_vec; i += (int64_t)gridDim.x * blockDim.x) {
    // every byte is touched exactly once per launch: streaming loads / stores
    const uint4 w = __ldcs(words + i);
    const uchar4 a = __ldcs(actions + i);
    const StepOut o0 = step_word(w.x, a.x, c), o1 = step_word(w.y, a.y, c), o2 = step_word(w.z, a.z, c),
                  o3 = step_word(w.w, a.w, c);
    __stcs(words + i, make_uint4(o0.word, o1.word, o2.word, o3.word));
    __stcs(rewards + i, make_float4(o0.reward, o1.reward, o2.reward, o3.reward));
    __stcs(flags + i, make_uchar4((unsigned char)o0.flags, (unsigned char)o1.flags, (unsigned char)o2.flags,
                                  (unsigned char)o3.flags));
    if (kObs) __stcs(obs_words + i, make_uint4(o0.obs_word, o1.obs_word, o2.obs_word, o3.obs_word));
  }
}

__global__ void __launch_bounds__(256) env_step_scalar(uint32_t* __restrict__ words, const uint8_t* __restrict__ actions,
                                                      float* __restrict__ rewards, uint8_t* __restrict__ flags,
                                                      uint32_t* __restrict__ obs_words, int64_t begin, int64_t n,
                                                      EnvCfg c) {
  for (int64_t i = begin + blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x) {
    StepOut o = step_word(words[i], actions[i], c);
    words[i] = o.word;
    rewards[i] = o.reward;
    flags[i] = (uint8_t)o.flags;
    if (obs_words) obs_words[i] = o.obs_word;
  }
}

__global__ void __launch_bounds__(256) env_step_random_vec4(uint4* __restrict__ words, uchar4* __restrict__ actions,
                                                           float4* __restrict__ rewards, uchar4* __restrict__ flags,
                                                           int64_t n_vec, EnvCfg c, uint32_t seed_lo, uint32_t seed_hi,
                                                           uint32_t step_lo, uint32_t step_hi) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n_vec; i += (int64_t)gridDim.x * blockDim.x) {
    const uint4 w = __ldcs(words + i);
    const Philox4 r = philox4x32_10((uint32_t)i, (uint32_t)(i >> 32), step_lo, step_hi, seed_lo, seed_hi);
    uint32_t a0, a1, a2, a3;
    const StepOut o0 = step_random_word(w.x, r.x, c, a0), o1 = step_random_word(w.y, r.y, c, a1),
                  o2 = step_random_word(w.z, r.z, c, a2), o3 = step_random_word(w.w, r.w, c, a3);
    __stcs(words + i, make_uint4(o0.word, o1.word, o2.word, o3.word));
    __stcs(actions + i, make_uchar4((unsigned char)a0, (unsigned char)a1, (unsigned char)a2, (unsigned char)a3));
    __stcs(rewards + i, make_float4(o0.reward, o1.reward, o2.reward, o3.reward));
    __stcs(flags + i, make_uchar4((unsigned char)o0.flags, (unsigned char)o1.flags, (unsigned char)o2.flags,
                                  (unsigned char)o3.flags));
  }
}

// Env e of a vec4 group i uses lane (e & 3) of the Philox block keyed by (i, step): the same
// stream as env_step_random_vec4 so fused and per-step stepping visit identical states.
__global__ void __launch_bounds__(256) env_rollout_random_vec4(uint4* __restrict__ words, int64_t n_vec, EnvCfg c,
                                                              int n_steps, uint32_t seed_lo, uint32_t seed_hi,
                                                              uint64_t step_index,
                                                              unsigned long long* __restrict__ counters) {
  unsigned long long goals = 0, truncs = 0, steps = 0, fold = 0;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n_vec; i += (int64_t)gridDim.x * blockDim.x) {
    uint4 w = words[i];
    for (int k = 0; k < n_steps; ++k) {
      uint64_t sidx = step_index + (uint64_t)k;
      Philox4 r = philox4x32_10((uint32_t)i, (uint32_t)(i >> 32), (uint32_t)sidx, (uint32_t)(sidx >> 32), seed_lo, seed_hi);
      uint32_t a0, a1, a2, a3;
      const StepOut o0 = step_random_word(w.x, r.x, c, a0), o1 = step_random_word(w.y, r.y, c, a1),
                    o2 = step_random_word(w.z, r.z, c, a2), o3 = step_random_word(w.w, r.w, c, a3);
      w = make_uint4(o0.word, o1.word, o2.word, o3.word);
      uint32_t fl = o0.flags | (o1.flags << 8) | (o2.flags << 16) | (o3.flags << 24);
      goals += __popc(fl & 0x04040404u);
      truncs += __popc(fl & 0x08080808u);
    }
    steps += 4ull * (unsigned long long)n_steps;
    fold ^= ((unsigned long long)(w.x ^ w.z) << 32) | (unsigned long long)(w.y ^ w.w);
    words[i] = w;
  }
  // warp-reduce, one atomic per warp per counter
  for (int off = 16; off; off >>= 1) {
    goals += __shfl_xor_sync(0xffffffffu, goals, off);
    truncs += __shfl_xor_sync(0xffffffffu, truncs, off);
    steps += __shfl_xor_sync(0xffffffffu, steps, off);
    fold ^= __shfl_xor_sync(0xffffffffu, fold, off);
  }
  if ((threadIdx.x & 31) == 0) {
    atomicAdd(&counters[0], steps);
    atomicAdd(&counters[1], goals);
    atomicAdd(&counters[2], truncs);
    atomicXor(&counters[3], fold);
  }
}

__global__ void __launch_bounds__(256) env_fill(uint32_t* __restrict__ words, int64_t n, uint32_t value) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    words[i] = value;
}

__device__ __forceinline__ uint32_t index_to_word(uint32_t idx, int n_disks) {
  uint32_t w = 0;
  for (int d = n_disks - 1; d >= 0; --d) {  // disk 0 is the most significant base-3 digit
    uint32_t q = idx / 3u;
    w |= (idx - 3u * q) << (2 * d);
    idx = q;
  }
  return w;
}

__global__ void __launch_bounds__(256) env_from_index(const uint32_t* __restrict__ index, uint32_t* __restrict__ words,
                                                     int64_t n, int n_disks) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    words[i] = index_to_word(index[i], n_disks);
}

__global__ void __launch_bounds__(256) env_to_index(const uint32_t* __restrict__ words, uint32_t* __restrict__ index,
                                                   int64_t n, int n_disks) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    uint32_t w = words[i], idx = 0;
    for (int d = 0; d < n_disks; ++d) idx = idx * 3u + ((w >> (2 * d)) & 3u);
    index[i] = idx;
  }
}

__global__ void __launch_bounds__(256) env_random_reset(uint32_t* __restrict__ words, int64_t n, int n_disks,
                                                       uint32_t n_states, uint32_t goal_index, uint32_t seed_lo,
                                                       uint32_t seed_hi, uint32_t ctr_lo, uint32_t ctr_hi) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    Philox4 r = philox4x32_10((uint32_t)i, (uint32_t)(i >> 32), ctr_lo, ctr_hi, seed_lo ^ 0x52455345u, seed_hi);
    // uniform over the n_states-1 non-goal states (same law as the rejection loop of :105-109)
    uint32_t idx = __umulhi(r.x, n_states - 1u);
    idx += (uint32_t)(idx >= goal_index);
    words[i] = index_to_word(idx, n_disks);
  }
}

__global__ void __launch_bounds__(256) env_legal_mask(const uint32_t* __restrict__ words, uint8_t* __restrict__ mask,
                                                     int64_t n, uint32_t even_mask, uint32_t state_mask) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    uint32_t k0, k1, k2;
    peg_keys(words[i] & state_mask, even_mask, k0, k1, k2);
    mask[i] = (uint8_t)legal_bits(k0, k1, k2);
  }
}

// One thread per output float so that stores are fully coalesced: obs[i, 3d+p] = [disk d on peg p].
__global__ void __launch_bounds__(256) env_onehot(const uint32_t* __restrict__ words, float* __restrict__ obs,
                                                 int64_t n, int n_disks) {
  const int width = 3 * n_disks;
  const int64_t total = n * width;
  for (int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; j < total; j += (int64_t)gridDim.x * blockDim.x) {
    int64_t i = j / width;
    int col = (int)(j - i * width);
    int d = col / 3, p = col - 3 * d;
    obs[j] = (((words[i] >> (2 * d)) & 3u) == (uint32_t)p) ? 1.0f : 0.0f;
  }
}

__global__ void __launch_bounds__(256) env_solver(const uint32_t* __restrict__ words, uint32_t* __restrict__ dist,
                                                 int64_t n, int n_disks, int goal_peg) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    uint32_t w = words[i], moves = 0, target = (uint32_t)goal_peg;
    for (int d = n_disks - 1; d >= 0; --d) {  // env/hanoi_utils.py:19-24, largest disk first
      uint32_t peg = (w >> (2 * d)) & 3u;
      if (peg != target) {
        moves += 1u << d;
        target = 3u - target - peg;
      }
    }
    dist[i] = moves;
  }
}

// ------------------------------------------------------------------------------ host side
int make_env_cfg(EnvCfg& c, int n_disks, int max_steps, int goal_peg, int auto_reset, uint32_t reset_word) {
  if (n_disks < 1 || n_disks > HMZ_MAX_DISKS)
    return fail(HMZ_ERR_UNSUPPORTED, "n_disks=%d outside [1, %d]", n_disks, HMZ_MAX_DISKS);
  if (goal_peg < 0 || goal_peg > 2) return fail(HMZ_ERR_INVALID, "goal_peg=%d outside [0, 2]", goal_peg);
  c.shift = 2 * n_disks;
  c.state_mask = (1u << c.shift) - 1u;
  c.even_mask = 0x55555555u & c.state_mask;
  uint64_t room = 1ull << (32 - c.shift);
  if (max_steps < 1 || (uint64_t)max_steps >= room)
    return fail(HMZ_ERR_UNSUPPORTED, "max_steps=%d does not fit the %d counter bits of the env word", max_steps,
                32 - c.shift);
  c.max_steps = (uint32_t)max_steps;
  c.goal_word = c.even_mask * (uint32_t)goal_peg;
  c.reset_word = reset_word;
  c.auto_reset = auto_reset;
  return HMZ_OK;
}

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
static bool aligned4(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 3u) == 0; }

}  // namespace hmz

using namespace hmz;

extern "C" {

int hmz_env_reset(uint32_t* words, int64_t n, uint32_t reset_word, void* stream) {
  ProfScope prof_scope(HMZ_PROF_OTHER, stream);
  if (n == 0) return HMZ_OK;
  if (!words || n < 0) return fail(HMZ_ERR_INVALID, "hmz_env_reset: null pointer or negative size");
  env_fill<<<grid_for(n, 256, 8), 256, 0, (cudaStream_t)stream>>>(words, n, reset_word);
  return check_launch("env_fill");
}

int hmz_env_from_index(const uint32_t* index, uint32_t* words, int64_t n, int n_disks, void* stream) {
  ProfScope prof_scope(HMZ_PROF_OTHER, stream);
  if (n == 0) return HMZ_OK;
  if (!index || !words || n < 0 || n_disks < 1 || n_disks > HMZ_MAX_DISKS)
    return fail(HMZ_ERR_INVALID, "hmz_env_from_index: bad arguments");
  env_from_index<<<grid_for(n, 256, 8), 256, 0, (cudaStream_t)stream>>>(index, words, n, n_disks);
  return check_launch("env_from_index");
}

int hmz_env_to_index(const uint32_t* words, uint32_t* index, int64_t n, int n_disks, void* stream) {
  ProfScope prof_scope(HMZ_PROF_OTHER, stream);
  if (n == 0) return HMZ_OK;
  if (!index || !words || n < 0 || n_disks < 1 || n_disks > HMZ_MAX_DISKS)
    return fail(HMZ_ERR_INVALID, "hmz_env_to_index: bad arguments");
  env_to_index<<<grid_for(n, 256, 8), 256, 0, (cudaStream_t)stream>>>(words, index, n, n_disks);
  return check_launch("env_to_index");
}

int hmz_env_random_reset(uint32_t* words, int64_t n, int n_disks, int goal_peg, uint64_t seed, uint64_t counter,
                         void* stream) {
  ProfScope prof_scope(HMZ_PROF_OTHER, stream);
  if (n == 0) return HMZ_OK;
  if (!words || n < 0 || n_disks < 1 || n_disks > HMZ_MAX_DISKS || goal_peg < 0 || goal_peg > 2)
    return fail(HMZ_ERR_INVALID, "hmz_env_random_reset: bad arguments");
  if (n == 0) return HMZ_OK;
  uint32_t n_states = 1, goal_index = 0;
  for (int d = 0; d < n_disks; ++d) {
    n_states *= 3u;
    goal_index = goal_index * 3u + (uint32_t)goal_peg;
  }
  env_random_reset<<<grid_for(n, 256, 8), 256, 0, (cudaStream_t)stream>>>(
      words, n, n_disks, n_states, goal_index, (uint32_t)seed, (uint32_t)(seed >> 32), (uint32_t)counter,
      (uint32_t)(counter >> 32));
  return check_launch("env_random_reset");
}

int hmz_env_step(uint32_t* words, const uint8_t* actions, float* rewards, uint8_t* flags, uint32_t* obs_words,
                 int64_t n, int n_disks, int max_steps, int goal_peg, int auto_reset, uint32_t reset_word,
                 void* stream) {
  ProfScope prof_scope(HMZ_PROF_ENV, stream);
  if (n == 0) return HMZ_OK;
  if (!words || !actions || !rewards || !flags || n < 0) return fail(HMZ_ERR_INVALID, "hmz_env_step: null pointer");
  EnvCfg c;
  if (int rc = make_env_cfg(c, n_disks, max_steps, goal_peg, auto_reset, reset_word)) return rc;
  if (n == 0) return HMZ_OK;
  cudaStream_t st = (cudaStream_t)stream;
  bool vec = aligned16(words) && aligned4(actions) && aligned16(rewards) && aligned4(flags) &&
             (!obs_words || aligned16(obs_words));
  int64_t n_vec = vec ? n / 4 : 0;
  if (n_vec > 0) {
    const unsigned grid = grid_for(n_vec, 256, 8);
    (obs_words ? env_step_vec4<true> : env_step_vec4<false>)<<<grid, 256, 0, st>>>(
        (uint4*)words, (const uchar4*)actions, (float4*)rewards, (uchar4*)flags, (uint4*)obs_words, n_vec, c);
    if (int rc = check_launch("env_step_vec4")) return rc;
  }
  if (n_vec * 4 < n) {
    env_step_scalar<<<grid_for(n - n_vec * 4, 256, 8), 256, 0, st>>>(words, actions, rewards, flags, obs_words,
                                                                    n_vec * 4, n, c);
    if (int rc = check_launch("env_step_scalar")) return rc;
  }
  return HMZ_OK;
}

int hmz_env_legal_mask(const uint32_t* words, uint8_t* mask, int64_t n, int n_disks, void* stream) {
  ProfScope prof_scope(HMZ_PROF_OTHER, stream);
  if (n == 0) return HMZ_OK;
  if (!words || !mask || n < 0 || n_disks < 1 || n_disks > HMZ_MAX_DISKS)
    return fail(HMZ_ERR_INVALID, "hmz_env_legal_mask: bad arguments");
  if (n == 0) return HMZ_OK;
  uint32_t state_mask = (1u << (2 * n_disks)) - 1u;
  env_legal_mask<<<grid_for(n, 256, 8), 256, 0, (cudaStream_t)stream>>>(words, mask, n, 0x55555555u & state_mask,
                                                                         state_mask);
  return check_launch("env_legal_mask");
}

int hmz_env_onehot(const uint32_t* words, float* obs, int64_t n, int n_disks, void* stream) {
  ProfScope prof_scope(HMZ_PROF_OTHER, stream);
  if (n == 0) return HMZ_OK;
  if (!words || !obs || n < 0 || n_disks < 1 || n_disks > HMZ_MAX_DISKS)
    return fail(HMZ_ERR_INVALID, "hmz_env_onehot: bad arguments");
  env_onehot<<<grid_for(n * 3 * n_disks, 256, 8), 256, 0, (cudaStream_t)stream>>>(words, obs, n, n_disks);
  return check_launch("env_onehot");
}

int hmz_env_solver_distance(const uint32_t* words, uint32_t* distance, int64_t n, int n_disks, int goal_peg,
                            void* stream) {
  ProfScope prof_scope(HMZ_PROF_OTHER, stream);
  if (n == 0) return HMZ_OK;
  if (!words || !distance || n < 0 || n_disks < 1 || n_disks > HMZ_MAX_DISKS || goal_peg < 0 || goal_peg > 2)
    return fail(HMZ_ERR_INVALID, "hmz_env_solver_distance: bad arguments");
  env_solver<<<grid_for(n, 256, 8), 256, 0, (cudaStream_t)stream>>>(words, distance, n, n_disks, goal_peg);
  return check_launch("env_solver");
}

int hmz_env_step_random(uint32_t* words, uint8_t* actions, float* rewards, uint8_t* flags, int64_t n, int n_disks,
                        int max_steps, int goal_peg, uint32_t reset_word, uint64_t seed, uint64_t step_index,
                        void* stream) {
  ProfScope prof_scope(HMZ_PROF_ENV, stream);
  if (n == 0) return HMZ_OK;
  if (!words || !actions || !rewards || !flags || n < 0)
    return fail(HMZ_ERR_INVALID, "hmz_env_step_random: null pointer");
  EnvCfg c;
  if (int rc = make_env_cfg(c, n_disks, max_steps, goal_peg, 1, reset_word)) return rc;
  if (n % 4 != 0 || !aligned16(words) || !aligned4(actions) || !aligned16(rewards) || !aligned4(flags))
    return fail(HMZ_ERR_INVALID, "hmz_env_step_random: n_envs must be a multiple of 4 and buffers 16-byte aligned");
  env_step_random_vec4<<<grid_for(n / 4, 256, 8), 256, 0, (cudaStream_t)stream>>>(
      (uint4*)words, (uchar4*)actions, (float4*)rewards, (uchar4*)flags, n / 4, c, (uint32_t)seed, (uint32_t)(seed >> 32),
      (uint32_t)step_index, (uint32_t)(step_index >> 32));
  return check_launch("env_step_random_vec4");
}

int hmz_env_rollout_random(uint32_t* words, int64_t n, int n_disks, int max_steps, int goal_peg, uint32_t reset_word,
                           int n_steps, uint64_t seed, uint64_t step_index, unsigned long long* counters,
                           void* stream) {
  ProfScope prof_scope(HMZ_PROF_ENV, stream);
  if (n == 0) return HMZ_OK;
  if (!words || !counters || n < 0 || n_steps < 0) return fail(HMZ_ERR_INVALID, "hmz_env_rollout_random: bad arguments");
  EnvCfg c;
  if (int rc = make_env_cfg(c, n_disks, max_steps, goal_peg, 1, reset_word)) return rc;
  if (n % 4 != 0 || !aligned16(words))
    return fail(HMZ_ERR_INVALID, "hmz_env_rollout_random: n_envs must be a multiple of 4 and words 16-byte aligned");
  if (n == 0 || n_steps == 0) return HMZ_OK;
  env_rollout_random_vec4<<<grid_for(n / 4, 256, 8), 256, 0, (cudaStream_t)stream>>>(
      (uint4*)words, n / 4, c, n_steps, (uint32_t)seed, (uint32_t)(seed >> 32), step_index, counters);
  return check_launch("env_rollout_random_vec4");
}

}  // extern "C"
