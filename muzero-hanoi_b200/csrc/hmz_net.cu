// MuZeroNet inference, float32 FFMA path (HMZ_MODE_FP32 — the parity mode, <= 1e-5 of the
// reference's float32 torch outputs) + weight packing + mode dispatch.
//
// Restates networks.py of the reference: initial_inference :71-94 (represent :124-127 +
// prediction :140-150), recurrent_inference :96-116 (dynamics :129-138 + prediction), the
// support transform :152-189 and normalize_h_state :191-196.
//
// One CTA evaluates 32 rows (searches) through the whole g + f chain: activations stay in shared
// memory TRANSPOSED ([feature][row]) so each thread's register tile reads its rows with one
// 128-bit LDS, weights ([in][out], read-only, L1/L2 resident: 412 KB for all CTAs) stream
// through the read-only path.  The tensor-core path (bf16, tcgen05) lives in hmz_net_tc.cu.
#include <cstring>
#include <vector>

#include "hmz_net.cuh"

namespace hmz {

constexpr int kRows = 32;       // rows (searches) per CTA
constexpr int kRowStride = 36;  // floats between consecutive features in the transposed tiles
constexpr int kNetThreads = 256;

// Y^T[n][m] = act(bias[n] + sum_k X^T[k][m] * Wt[k][n] (+ Wrow[sel[m]][n]))   for a 32-row tile.
// Register tile TM x TN per thread; row groups vary fastest across lanes so that the X reads of a
// warp are one contiguous 128-byte span and the W reads coalesce.
template <int K, int NPAD, int TM, int TN, bool RELU, bool ROWBIAS>
__device__ __forceinline__ void dense_T(const float* __restrict__ xsT, const float* __restrict__ Wt,
                                        const float* __restrict__ bias, float* __restrict__ ysT,
                                        const float* __restrict__ Wrow, const int* __restrict__ sel) {
  static_assert(TM % 4 == 0 && (TN == 2 || TN == 4), "tile shape");
  constexpr int RG = kRows / TM, CG = NPAD / TN, TILES = RG * CG;
  for (int tile = threadIdx.x; tile < TILES; tile += kNetThreads) {
    const int rg = tile % RG, cg = tile / RG;
    const int m0 = rg * TM, n0 = cg * TN;
    float acc[TM][TN];
#pragma unroll
    for (int j = 0; j < TN; ++j) {
      const float b = __ldg(bias + n0 + j);
#pragma unroll
      for (int i = 0; i < TM; ++i) acc[i][j] = ROWBIAS ? b + __ldg(Wrow + sel[m0 + i] * NPAD + n0 + j) : b;
    }
#pragma unroll 4
    for (int k = 0; k < K; ++k) {
      float x[TM], w[TN];
#pragma unroll
      for (int i = 0; i < TM; i += 4) {
        const float4 t = *reinterpret_cast<const float4*>(xsT + k * kRowStride + m0 + i);
        x[i] = t.x; x[i + 1] = t.y; x[i + 2] = t.z; x[i + 3] = t.w;
      }
      if (TN == 4) {
        const float4 t = __ldg(reinterpret_cast<const float4*>(Wt + k * NPAD + n0));
        w[0] = t.x; w[1] = t.y; w[2] = t.z; w[3] = t.w;
      } else {
        const float2 t = __ldg(reinterpret_cast<const float2*>(Wt + k * NPAD + n0));
        w[0] = t.x; w[1] = t.y;
      }
#pragma unroll
      for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(x[i], w[j], acc[i][j]);
    }
#pragma unroll
    for (int j = 0; j < TN; ++j)
#pragma unroll
      for (int i = 0; i < TM; i += 4) {
        float4 t = make_float4(acc[i][j], acc[i + 1][j], acc[i + 2][j], acc[i + 3][j]);
        if (RELU) t = make_float4(fmaxf(t.x, 0.f), fmaxf(t.y, 0.f), fmaxf(t.z, 0.f), fmaxf(t.w, 0.f));
        *reinterpret_cast<float4*>(ysT + (n0 + j) * kRowStride + m0 + i) = t;
      }
  }
}

struct NetSmem {
  float x[kLatent * kRowStride];     // input latent (transposed)
  float hid[kHidden * kRowStride];   // hidden layer of whichever MLP is running
  float raw[kLatent * kRowStride];   // un-normalised new latent (reward head input, networks.py:131-132)
  float hn[kLatent * kRowStride];    // min-max normalised latent
  float lg[kSupportPad * kRowStride];  // head logits
  int sel[kRows];                    // action per row
  uint32_t word[kRows];              // env word per row (initial inference)
};

// normalize_h_state (networks.py:191-196), one lane per row, then the row-major latent store.
__device__ __forceinline__ void normalise_rows(NetSmem& s) {
  if (threadIdx.x < kRows) {
    const int m = threadIdx.x;
    float mn = s.raw[m], mx = s.raw[m];
#pragma unroll 8
    for (int k = 1; k < kLatent; ++k) {
      const float t = s.raw[k * kRowStride + m];
      mn = fminf(mn, t);
      mx = fmaxf(mx, t);
    }
    const float den = __fadd_rn(__fsub_rn(mx, mn), 1e-8f);
#pragma unroll 8
    for (int k = 0; k < kLatent; ++k)
      s.hn[k * kRowStride + m] = __fdiv_rn(__fsub_rn(s.raw[k * kRowStride + m], mn), den);
  }
}

__device__ __forceinline__ void store_latent_rows(const NetSmem& s, void* lat_out, int64_t out_rows_per_item,
                                                  int64_t out_row, int latent_dtype, int64_t row0, int64_t n) {
  const int m = threadIdx.x & 31, c = threadIdx.x >> 5;  // lane <-> row, warp <-> 8-feature chunk
  const int64_t item = row0 + m;
  if (item >= n) return;
  const int64_t orow = item * out_rows_per_item + out_row;
  float t[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) t[j] = s.hn[(c * 8 + j) * kRowStride + m];
  if (latent_dtype == HMZ_LATENT_F32) {
    float4* dst = reinterpret_cast<float4*>(reinterpret_cast<float*>(lat_out) + orow * kLatent + c * 8);
    dst[0] = make_float4(t[0], t[1], t[2], t[3]);
    dst[1] = make_float4(t[4], t[5], t[6], t[7]);
  } else {
    uint32_t pk[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const uint32_t lo = __float_as_uint(t[2 * j]), hi = __float_as_uint(t[2 * j + 1]);
      // round-to-nearest-even float32 -> bf16
      const uint32_t l16 = (lo + 0x7FFFu + ((lo >> 16) & 1u)) >> 16, h16 = (hi + 0x7FFFu + ((hi >> 16) & 1u)) >> 16;
      pk[j] = l16 | (h16 << 16);
    }
    *reinterpret_cast<uint4*>(reinterpret_cast<uint16_t*>(lat_out) + orow * kLatent + c * 8) =
        make_uint4(pk[0], pk[1], pk[2], pk[3]);
  }
}

// prediction() heads on the normalised latent + (optionally) the reward head on the raw latent.
template <bool kReward>
__device__ __forceinline__ void run_heads(NetSmem& s, const float* __restrict__ W, float* __restrict__ r,
                                          float* __restrict__ p, float* __restrict__ v, int64_t row0, int64_t n) {
  using L = Fp32Layout;
  const int m = threadIdx.x;
  const bool row_ok = (m < kRows) && (row0 + m < n);
  if (kReward) {
    dense_T<kLatent, kHidden, 8, 4, true, false>(s.raw, W + L::rwd_w1, W + L::rwd_b1, s.hid, nullptr, nullptr);
    __syncthreads();
    dense_T<kHidden, kSupportPad, 4, 2, false, false>(s.hid, W + L::rwd_w2, W + L::rwd_b2, s.lg, nullptr, nullptr);
    __syncthreads();
    if (row_ok) r[row0 + m] = support_to_scalar([&](int i) { return s.lg[i * kRowStride + m]; });
  }
  dense_T<kLatent, kHidden, 8, 4, true, false>(s.hn, W + L::pol_w1, W + L::pol_b1, s.hid, nullptr, nullptr);
  __syncthreads();
  dense_T<kHidden, kPolicyPad, 4, 2, false, false>(s.hid, W + L::pol_w2, W + L::pol_b2, s.lg, nullptr, nullptr);
  __syncthreads();
  if (row_ok) {  // F.softmax(pi_logits) (networks.py:83,109)
    float lg[kActions], mx = s.lg[m];
#pragma unroll
    for (int a = 0; a < kActions; ++a) {
      lg[a] = s.lg[a * kRowStride + m];
      mx = fmaxf(mx, lg[a]);
    }
    float den = 0.f;
#pragma unroll
    for (int a = 0; a < kActions; ++a) {
      lg[a] = expf(lg[a] - mx);
      den += lg[a];
    }
#pragma unroll
    for (int a = 0; a < kActions; ++a) p[(row0 + m) * kActions + a] = __fdiv_rn(lg[a], den);
  }
  dense_T<kLatent, kHidden, 8, 4, true, false>(s.hn, W + L::val_w1, W + L::val_b1, s.hid, nullptr, nullptr);
  __syncthreads();
  dense_T<kHidden, kSupportPad, 4, 2, false, false>(s.hid, W + L::val_w2, W + L::val_b2, s.lg, nullptr, nullptr);
  __syncthreads();
  if (row_ok) v[row0 + m] = support_to_scalar([&](int i) { return s.lg[i * kRowStride + m]; });
}

// Heterogeneous batches (hmz_multi_t): the weight set of this CTA's 256-row block (kRows divides 256).
__device__ __forceinline__ const float* set_weights(const float* W, const uint16_t* block_set, int64_t weight_stride) {
  if (block_set == nullptr) return W;
  const int64_t block = (int64_t)blockIdx.x * kRows / 256;
  return reinterpret_cast<const float*>(reinterpret_cast<const char*>(W) + (int64_t)block_set[block] * weight_stride);
}

__global__ void __launch_bounds__(kNetThreads, 3)
net_recurrent_fp32(const float* __restrict__ W_base, const uint16_t* __restrict__ block_set, int64_t weight_stride,
                   const void* __restrict__ lat_in, int64_t in_rows_per_item,
                   const uint16_t* __restrict__ in_row, const uint8_t* __restrict__ actions, void* lat_out,
                   int64_t out_rows_per_item, int64_t out_row, int latent_dtype, float* __restrict__ r,
                   float* __restrict__ p, float* __restrict__ v, int64_t n) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  NetSmem& s = *reinterpret_cast<NetSmem*>(smem_raw);
  using L = Fp32Layout;
  const int64_t row0 = (int64_t)blockIdx.x * kRows;
  const float* __restrict__ W = set_weights(W_base, block_set, weight_stride);
  {  // gather the parent latents: lane <-> row, warp <-> 8-feature chunk
    const int m = threadIdx.x & 31, c = threadIdx.x >> 5;
    int64_t item = row0 + m;
    if (item >= n) item = n - 1;
    const int64_t irow = item * in_rows_per_item + (in_row ? (int64_t)in_row[item] : 0);
    float t[8];
    if (latent_dtype == HMZ_LATENT_F32) {
      const float4* src = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(lat_in) + irow * kLatent + c * 8);
      const float4 a = src[0], b = src[1];
      t[0] = a.x; t[1] = a.y; t[2] = a.z; t[3] = a.w; t[4] = b.x; t[5] = b.y; t[6] = b.z; t[7] = b.w;
    } else {
      const uint4 q = *reinterpret_cast<const uint4*>(reinterpret_cast<const uint16_t*>(lat_in) + irow * kLatent + c * 8);
      const uint32_t pk[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        t[2 * j] = __uint_as_float(pk[j] << 16);
        t[2 * j + 1] = __uint_as_float(pk[j] & 0xFFFF0000u);
      }
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) s.x[(c * 8 + j) * kRowStride + m] = t[j];
    if (c == 0) {
      const int a = actions[item];
      s.sel[m] = a < kActions ? a : kActions - 1;
    }
  }
  __syncthreads();
  // dynamics (networks.py:129-138): Linear(70,256)+ReLU on cat[h, onehot(a)] — the one-hot part is
  // row (64 + a) of the transposed weight, added as a per-row bias — then Linear(256,64).
  dense_T<kLatent, kHidden, 8, 4, true, true>(s.x, W + L::dyn_w1, W + L::dyn_b1, s.hid,
                                              W + L::dyn_w1 + kLatent * kHidden, s.sel);
  __syncthreads();
  dense_T<kHidden, kLatent, 4, 2, false, false>(s.hid, W + L::dyn_w2, W + L::dyn_b2, s.raw, nullptr, nullptr);
  __syncthreads();
  normalise_rows(s);
  __syncthreads();
  store_latent_rows(s, lat_out, out_rows_per_item, out_row, latent_dtype, row0, n);
  run_heads<true>(s, W, r, p, v, row0, n);
}

__global__ void __launch_bounds__(kNetThreads, 3)
net_initial_fp32(const float* __restrict__ W_base, const uint16_t* __restrict__ block_set, int64_t weight_stride, int n_disks, const uint32_t* __restrict__ words,
                 const float* __restrict__ obs, void* lat_out, int64_t out_rows_per_item, int latent_dtype,
                 float* __restrict__ p0, float* __restrict__ v0, int64_t n) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  NetSmem& s = *reinterpret_cast<NetSmem*>(smem_raw);
  using L = Fp32Layout;
  const int64_t row0 = (int64_t)blockIdx.x * kRows;
  const float* __restrict__ W = set_weights(W_base, block_set, weight_stride);
  const int width = 3 * n_disks;
  const float* w1 = W + L::rep_w1;
  const float* b1 = W + L::rep_b1(n_disks);
  if (words) {
    if (threadIdx.x < kRows) {
      int64_t item = row0 + threadIdx.x;
      s.word[threadIdx.x] = words[item < n ? item : n - 1];
    }
  } else {  // general float observation (noise_injection_comparison.py:25-31 feeds non-one-hot vectors)
    for (int idx = threadIdx.x; idx < kRows * width; idx += kNetThreads) {
      const int m = idx / width, k = idx - m * width;
      int64_t item = row0 + m;
      if (item >= n) item = n - 1;
      s.x[k * kRowStride + m] = obs[item * width + k];  // width <= 36 <= kLatent rows of s.x
    }
  }
  __syncthreads();
  {  // representation layer 1 (Linear(3N,256)+ReLU): thread <-> hidden unit
    const int nn = threadIdx.x;
    const float b = __ldg(b1 + nn);
    if (words) {  // one-hot input: a sum of N weight rows
      for (int m = 0; m < kRows; ++m) {
        const uint32_t wd = s.word[m];
        float acc = b;
        for (int d = 0; d < n_disks; ++d) acc += __ldg(w1 + (3 * d + ((wd >> (2 * d)) & 3u)) * kHidden + nn);
        s.hid[nn * kRowStride + m] = fmaxf(acc, 0.f);
      }
    } else {
      float acc[kRows];
#pragma unroll
      for (int m = 0; m < kRows; ++m) acc[m] = b;
      for (int k = 0; k < width; ++k) {
        const float w = __ldg(w1 + k * kHidden + nn);
#pragma unroll
        for (int m = 0; m < kRows; ++m) acc[m] = fmaf(s.x[k * kRowStride + m], w, acc[m]);
      }
#pragma unroll
      for (int m = 0; m < kRows; ++m) s.hid[nn * kRowStride + m] = fmaxf(acc[m], 0.f);
    }
  }
  __syncthreads();
  dense_T<kHidden, kLatent, 4, 2, false, false>(s.hid, W + L::rep_w2(n_disks), W + L::rep_b2(n_disks), s.raw, nullptr,
                                                nullptr);
  __syncthreads();
  normalise_rows(s);
  __syncthreads();
  store_latent_rows(s, lat_out, out_rows_per_item, 0, latent_dtype, row0, n);
  run_heads<false>(s, W, nullptr, p0, v0, row0, n);
}

// ------------------------------------------------------------------------------ packing
// state_dict order: {representation, dynamic, rwd, policy, value} x {0.weight, 0.bias, 2.weight, 2.bias};
// torch Linear weights are [out][in] row-major.
static void transpose_into(float* dst, const float* w, int out, int in, int out_pad) {
  for (int k = 0; k < in; ++k)
    for (int o = 0; o < out_pad; ++o) dst[k * out_pad + o] = o < out ? w[o * in + k] : 0.0f;
}

static void copy_bias(float* dst, const float* b, int out, int out_pad) {
  for (int o = 0; o < out_pad; ++o) dst[o] = o < out ? b[o] : 0.0f;
}

void pack_fp32(const float* const* t, int n_disks, float* out) {
  using L = Fp32Layout;
  const int in0 = 3 * n_disks;
  transpose_into(out + L::rep_w1, t[0], kHidden, in0, kHidden);
  copy_bias(out + L::rep_b1(n_disks), t[1], kHidden, kHidden);
  transpose_into(out + L::rep_w2(n_disks), t[2], kLatent, kHidden, kLatent);
  copy_bias(out + L::rep_b2(n_disks), t[3], kLatent, kLatent);
  transpose_into(out + L::dyn_w1, t[4], kHidden, kLatent + kActions, kHidden);
  copy_bias(out + L::dyn_b1, t[5], kHidden, kHidden);
  transpose_into(out + L::dyn_w2, t[6], kLatent, kHidden, kLatent);
  copy_bias(out + L::dyn_b2, t[7], kLatent, kLatent);
  transpose_into(out + L::rwd_w1, t[8], kHidden, kLatent, kHidden);
  copy_bias(out + L::rwd_b1, t[9], kHidden, kHidden);
  transpose_into(out + L::rwd_w2, t[10], kSupport, kHidden, kSupportPad);
  copy_bias(out + L::rwd_b2, t[11], kSupport, kSupportPad);
  transpose_into(out + L::pol_w1, t[12], kHidden, kLatent, kHidden);
  copy_bias(out + L::pol_b1, t[13], kHidden, kHidden);
  transpose_into(out + L::pol_w2, t[14], kActions, kHidden, kPolicyPad);
  copy_bias(out + L::pol_b2, t[15], kActions, kPolicyPad);
  transpose_into(out + L::val_w1, t[16], kHidden, kLatent, kHidden);
  copy_bias(out + L::val_b1, t[17], kHidden, kHidden);
  transpose_into(out + L::val_w2, t[18], kSupport, kHidden, kSupportPad);
  copy_bias(out + L::val_b2, t[19], kSupport, kSupportPad);
}


static int ensure_smem_optin() {
  static thread_local int done_dev = -1;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return fail(HMZ_ERR_CUDA, "cudaGetDevice failed (no CUDA device?)");
  if (done_dev == dev) return HMZ_OK;
  cudaError_t e = cudaFuncSetAttribute(net_recurrent_fp32, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(NetSmem));
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(net_initial_fp32, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(NetSmem));
  if (e != cudaSuccess) return fail(HMZ_ERR_CUDA, "cudaFuncSetAttribute(net_*_fp32): %s", cudaGetErrorString(e));
  done_dev = dev;
  return HMZ_OK;
}

}  // namespace hmz

using namespace hmz;

extern "C" {

int hmz_debug_tc_timeline(unsigned long long* host_out) { return tc_debug_read_timeline(host_out); }
int hmz_debug_x3_timeline(unsigned long long* host_out) { return x3::debug_read_timeline(host_out); }

int64_t hmz_weights_packed_bytes(int n_disks, int mode) {
  if (n_disks < 1 || n_disks > HMZ_MAX_DISKS) return -1;
  if (mode == HMZ_MODE_FP32) return (int64_t)Fp32Layout::total(n_disks) * 4;
  if (mode == HMZ_MODE_BF16) return tc_packed_bytes(n_disks);
  if (mode == HMZ_MODE_FP32X3) return x3::packed_bytes(n_disks);
  return -1;
}

int hmz_weights_pack(const float* const* host_tensors, int n_disks, int mode, void* host_out) {
  if (!host_tensors || !host_out || n_disks < 1 || n_disks > HMZ_MAX_DISKS)
    return fail(HMZ_ERR_INVALID, "hmz_weights_pack: bad arguments");
  for (int i = 0; i < 20; ++i)
    if (!host_tensors[i]) return fail(HMZ_ERR_INVALID, "hmz_weights_pack: tensor %d is null", i);
  if (mode == HMZ_MODE_FP32) {
    pack_fp32(host_tensors, n_disks, (float*)host_out);
    return HMZ_OK;
  }
  if (mode == HMZ_MODE_BF16) {
    tc_pack(host_tensors, n_disks, host_out);
    return HMZ_OK;
  }
  if (mode == HMZ_MODE_FP32X3) {
    x3::pack(host_tensors, n_disks, host_out);
    return HMZ_OK;
  }
  return fail(HMZ_ERR_INVALID, "hmz_weights_pack: unknown mode %d", mode);
}

int hmz_net_initial(const void* weights, int mode, int n_disks, const uint32_t* words, const float* obs,
                    void* latents_out, int64_t out_rows_per_item, int latent_dtype, float* p0, float* v0, int64_t n,
                    void* stream) {
  ProfScope prof_scope(HMZ_PROF_NET_INITIAL, stream);
  return net_initial_sets(weights, nullptr, 0, mode, n_disks, words, obs, latents_out, out_rows_per_item, latent_dtype, p0, v0, n,
                          stream);
}

int hmz_net_initial_multi(const void* weights, const hmz_multi_t* m, int mode, const uint32_t* words, void* latents_out,
                          int64_t out_rows_per_item, int latent_dtype, float* p0, float* v0, int64_t n, void* stream) {
  ProfScope prof_scope(HMZ_PROF_NET_INITIAL, stream);
  if (int rc = check_multi(m, n, mode, 0, false, "hmz_net_initial_multi")) return rc;
  if (n > 0 && !words) return fail(HMZ_ERR_INVALID, "hmz_net_initial_multi: null words");
  return net_initial_sets(weights, m->block_set, m->weight_stride, mode, m->n_disks, words, nullptr, latents_out, out_rows_per_item,
                          latent_dtype, p0, v0, n, stream);
}

int hmz_net_recurrent(const void* weights, int mode, const void* latents_in, int64_t in_rows_per_item,
                      const uint16_t* in_row, const uint8_t* actions, void* latents_out, int64_t out_rows_per_item,
                      int64_t out_row, int latent_dtype, float* r, float* p, float* v, int64_t n, void* stream) {
  ProfScope prof_scope(HMZ_PROF_NET_RECURRENT, stream);
  return net_recurrent_sets(weights, nullptr, 0, true, mode, latents_in, in_rows_per_item, in_row, actions, latents_out,
                            out_rows_per_item, out_row, latent_dtype, r, p, v, n, stream);
}

}  // extern "C"

namespace hmz {

int check_multi(const hmz_multi_t* m, int64_t n_searches, int mode, int n_records, bool need_budget, const char* who) {
  if (!m) return fail(HMZ_ERR_INVALID, "%s: null hmz_multi_t", who);
  if (n_searches < 0 || n_searches % 256 != 0)
    return fail(HMZ_ERR_INVALID, "%s: n_searches=%lld is not a multiple of 256", who, (long long)n_searches);
  if (m->n_sets < 1) return fail(HMZ_ERR_INVALID, "%s: n_sets=%d < 1", who, m->n_sets);
  if (mode >= 0) {  // the entry point reads weights (mode < 0: the root policy reads none)
    const int64_t need = hmz_weights_packed_bytes(m->n_disks, mode);
    if (need < 0) return fail(HMZ_ERR_INVALID, "%s: no packed layout for n_disks=%d, mode=%d", who, m->n_disks, mode);
    // >= one packed set, and a multiple of 256 bytes so that every set keeps the alignment of the blob's bulk copies
    if (m->weight_stride < need || m->weight_stride % 256 != 0)
      return fail(HMZ_ERR_INVALID, "%s: weight_stride=%lld must be >= %lld and a multiple of 256", who, (long long)m->weight_stride,
                  (long long)need);
    if (n_searches > 0 && !m->block_set) return fail(HMZ_ERR_INVALID, "%s: null block_set", who);
  }
  if (!need_budget || n_searches == 0) return HMZ_OK;
  if (!m->budget || !m->host_block_budget) return fail(HMZ_ERR_INVALID, "%s: null budget / host_block_budget", who);
  const int64_t blocks = n_searches / 256;
  for (int64_t k = 0; k < blocks; ++k) {
    const int32_t b = m->host_block_budget[k];
    if (b < 1 || b + 1 > n_records)
      return fail(HMZ_ERR_INVALID, "%s: block %lld budget %d outside [1, n_records - 1 = %d]", who, (long long)k, b, n_records - 1);
    if (k > 0 && b > m->host_block_budget[k - 1])
      return fail(HMZ_ERR_INVALID, "%s: block budgets must not increase (block %lld: %d after %d)", who, (long long)k, b,
                  m->host_block_budget[k - 1]);
  }
  return HMZ_OK;
}

int net_initial_sets(const void* weights, const uint16_t* block_set, int64_t weight_stride, int mode, int n_disks,
                     const uint32_t* words, const float* obs, void* latents_out, int64_t out_rows_per_item, int latent_dtype,
                     float* p0, float* v0, int64_t n, void* stream) {
  if (n == 0) return HMZ_OK;
  if (!weights || (!words && !obs) || !latents_out || !p0 || !v0 || n < 0 || n_disks < 1 || n_disks > HMZ_MAX_DISKS ||
      out_rows_per_item < 1 || (latent_dtype != HMZ_LATENT_F32 && latent_dtype != HMZ_LATENT_BF16))
    return fail(HMZ_ERR_INVALID, "hmz_net_initial: bad arguments");
  // HMZ_MODE_BF16 / HMZ_MODE_FP32X3 blobs embed a float32 copy of the weights behind the tensor-core section.
  if (mode != HMZ_MODE_FP32 && mode != HMZ_MODE_BF16 && mode != HMZ_MODE_FP32X3) return fail(HMZ_ERR_INVALID, "hmz_net_initial: unknown mode %d", mode);
  // throughput mode with packed env words: the tcgen05 kernel (bf16 representation + policy + value);
  // float observations (drop-in B = 1 views, arbitrary input vectors) keep the float32 kernel below
  if (mode == HMZ_MODE_BF16 && words != nullptr)
    return tc_net_initial(weights, n_disks, words, latents_out, out_rows_per_item, latent_dtype, p0, v0, n, (cudaStream_t)stream,
                          block_set, weight_stride);
  if (mode == HMZ_MODE_FP32X3 && words != nullptr)  // float32 accuracy on tcgen05, like the recurrent inference of this mode
    return x3::net_initial(weights, n_disks, words, latents_out, out_rows_per_item, latent_dtype, p0, v0, n, (cudaStream_t)stream,
                           block_set, weight_stride);
  if (int rc = ensure_smem_optin()) return rc;
  const unsigned grid = (unsigned)((n + kRows - 1) / kRows);
  const int64_t w32_off = mode == HMZ_MODE_BF16 ? tc_fp32_offset_bytes() : (mode == HMZ_MODE_FP32X3 ? x3::fp32_offset_bytes() : 0);
  const float* w32 = reinterpret_cast<const float*>(reinterpret_cast<const char*>(weights) + w32_off);
  net_initial_fp32<<<grid, kNetThreads, sizeof(NetSmem), (cudaStream_t)stream>>>(
      w32, block_set, weight_stride, n_disks, words, obs, latents_out, out_rows_per_item, latent_dtype, p0, v0, n);
  return check_launch("net_initial_fp32");
}

int net_recurrent_sets(const void* weights, const uint16_t* block_set, int64_t weight_stride, bool allow_head_split, int mode,
                       const void* latents_in, int64_t in_rows_per_item, const uint16_t* in_row, const uint8_t* actions,
                       void* latents_out, int64_t out_rows_per_item, int64_t out_row, int latent_dtype, float* r, float* p, float* v,
                       int64_t n, void* stream) {
  if (n == 0) return HMZ_OK;
  if (!weights || !latents_in || !actions || !latents_out || !r || !p || !v || n < 0 || in_rows_per_item < 1 ||
      out_rows_per_item < 1 || out_row < 0 || out_row >= out_rows_per_item ||
      (latent_dtype != HMZ_LATENT_F32 && latent_dtype != HMZ_LATENT_BF16))
    return fail(HMZ_ERR_INVALID, "hmz_net_recurrent: bad arguments");
  if (mode == HMZ_MODE_BF16)
    return tc_net_recurrent(weights, latents_in, in_rows_per_item, in_row, actions, latents_out, out_rows_per_item,
                            out_row, latent_dtype, r, p, v, n, (cudaStream_t)stream, block_set, weight_stride, allow_head_split);
  if (mode == HMZ_MODE_FP32X3)
    return x3::net_recurrent(weights, latents_in, in_rows_per_item, in_row, actions, latents_out, out_rows_per_item, out_row,
                             latent_dtype, r, p, v, n, (cudaStream_t)stream, block_set, weight_stride, allow_head_split);
  if (mode != HMZ_MODE_FP32) return fail(HMZ_ERR_INVALID, "hmz_net_recurrent: unknown mode %d", mode);
  if (int rc = ensure_smem_optin()) return rc;
  const unsigned grid = (unsigned)((n + kRows - 1) / kRows);
  net_recurrent_fp32<<<grid, kNetThreads, sizeof(NetSmem), (cudaStream_t)stream>>>(
      (const float*)weights, block_set, weight_stride, latents_in, in_rows_per_item, in_row, actions, latents_out, out_rows_per_item, out_row,
      latent_dtype, r, p, v, n);
  return check_launch("net_recurrent_fp32");
}

}  // namespace hmz
