// Weight-blob layouts and the float32 epilogue math of MuZeroNet inference, shared by the FFMA
// (parity) and tcgen05 (throughput) kernels.
#pragma once
#include "hmz_common.cuh"

namespace hmz {

constexpr int kLatent = HMZ_LATENT;    // 64
constexpr int kHidden = HMZ_HIDDEN;    // 256
constexpr int kSupport = HMZ_SUPPORT;  // 33
constexpr int kActions = HMZ_N_ACTIONS;
constexpr int kSupportPad = 36;  // 33 logits padded to a multiple of 4 (zero weights)
constexpr int kPolicyPad = 8;    // 6 logits padded to 8

// ---- float32 blob (HMZ_MODE_FP32): every Linear stored TRANSPOSED, [in][out_padded], so that the
// threads of a warp read consecutive output columns.  representation_net comes last so that the
// offsets of the recurrent path do not depend on the number of disks.
struct Fp32Layout {
  static constexpr int dyn_w1 = 0;                                   // [70][256]
  static constexpr int dyn_b1 = dyn_w1 + (kLatent + kActions) * kHidden;
  static constexpr int dyn_w2 = dyn_b1 + kHidden;                    // [256][64]
  static constexpr int dyn_b2 = dyn_w2 + kHidden * kLatent;
  static constexpr int rwd_w1 = dyn_b2 + kLatent;                    // [64][256]
  static constexpr int rwd_b1 = rwd_w1 + kLatent * kHidden;
  static constexpr int rwd_w2 = rwd_b1 + kHidden;                    // [256][36]
  static constexpr int rwd_b2 = rwd_w2 + kHidden * kSupportPad;
  static constexpr int pol_w1 = rwd_b2 + kSupportPad;                // [64][256]
  static constexpr int pol_b1 = pol_w1 + kLatent * kHidden;
  static constexpr int pol_w2 = pol_b1 + kHidden;                    // [256][8]
  static constexpr int pol_b2 = pol_w2 + kHidden * kPolicyPad;
  static constexpr int val_w1 = pol_b2 + kPolicyPad;                 // [64][256]
  static constexpr int val_b1 = val_w1 + kLatent * kHidden;
  static constexpr int val_w2 = val_b1 + kHidden;                    // [256][36]
  static constexpr int val_b2 = val_w2 + kHidden * kSupportPad;
  static constexpr int rep_w1 = val_b2 + kSupportPad;                // [3N][256]
  __host__ __device__ static constexpr int rep_b1(int n_disks) { return rep_w1 + 3 * n_disks * kHidden; }
  __host__ __device__ static constexpr int rep_w2(int n_disks) { return rep_b1(n_disks) + kHidden; }  // [256][64]
  __host__ __device__ static constexpr int rep_b2(int n_disks) { return rep_w2(n_disks) + kHidden * kLatent; }
  __host__ __device__ static constexpr int total(int n_disks) { return rep_b2(n_disks) + kLatent; }
};

// host: packs the 20 state_dict tensors into the float32 blob (hmz_net.cu)
void pack_fp32(const float* const* tensors, int n_disks, float* out);
// tensor-core path (hmz_net_tc.cu)
int64_t tc_packed_bytes(int n_disks);
int64_t tc_fp32_offset_bytes();
int tc_debug_read_timeline(unsigned long long* host_out);
void tc_pack(const float* const* tensors, int n_disks, void* out);
int tc_net_initial(const void* weights, int n_disks, const uint32_t* words, void* lat_out, int64_t out_rows_per_item,
                   int latent_dtype, float* p0, float* v0, int64_t n, cudaStream_t stream, const uint16_t* block_set = nullptr,
                   int64_t weight_stride = 0);
int tc_net_recurrent(const void* weights, const void* lat_in, int64_t in_rows_per_item, const uint16_t* in_row,
                     const uint8_t* actions, void* lat_out, int64_t out_rows_per_item, int64_t out_row,
                     int latent_dtype, float* r, float* p, float* v, int64_t n, cudaStream_t stream,
                     const uint16_t* block_set, int64_t weight_stride, bool allow_head_split);

// float32-accurate tensor-core path (hmz_net_x3.cu, HMZ_MODE_FP32X3): split section + the float32 blob behind it
namespace x3 {
int64_t packed_bytes(int n_disks);
int64_t fp32_offset_bytes();
void pack(const float* const* tensors, int n_disks, void* out);
int net_recurrent(const void* weights, const void* lat_in, int64_t in_rows_per_item, const uint16_t* in_row,
                  const uint8_t* actions, void* lat_out, int64_t out_rows_per_item, int64_t out_row, int latent_dtype,
                  float* r, float* p, float* v, int64_t n, cudaStream_t stream, const uint16_t* block_set,
                  int64_t weight_stride, bool allow_head_split);
int net_initial(const void* weights, int n_disks, const uint32_t* words, void* lat_out, int64_t out_rows_per_item,
                int latent_dtype, float* p0, float* v0, int64_t n, cudaStream_t stream, const uint16_t* block_set = nullptr,
                int64_t weight_stride = 0);
int debug_read_timeline(unsigned long long* host_out);
}  // namespace x3

// Both inferences with an optional weight set per 256-row block (hmz_multi_t): block_set == nullptr is the plain call;
// otherwise block k of the batch uses weights + block_set[k] * weight_stride (hmz_net.cu).  allow_head_split: the tensor-core
// kernels may spread a small batch over three CTAs per tile (one head each); hmz_search_run forbids it while several stream
// groups share the machine, as the other groups' launches want the idle SMs.
int net_initial_sets(const void* weights, const uint16_t* block_set, int64_t weight_stride, int mode, int n_disks,
                     const uint32_t* words, const float* obs, void* latents_out, int64_t out_rows_per_item, int latent_dtype,
                     float* p0, float* v0, int64_t n, void* stream);
int net_recurrent_sets(const void* weights, const uint16_t* block_set, int64_t weight_stride, bool allow_head_split, int mode,
                       const void* latents_in, int64_t in_rows_per_item, const uint16_t* in_row, const uint8_t* actions,
                       void* latents_out, int64_t out_rows_per_item, int64_t out_row, int latent_dtype, float* r, float* p, float* v,
                       int64_t n, void* stream);
// Argument checks of the hmz_multi_t entry points (before any CUDA call); need_budget: budget, host_block_budget and
// their bounds against n_records are checked too.
int check_multi(const hmz_multi_t* m, int64_t n_searches, int mode, int n_records, bool need_budget, const char* who);

// ---- epilogue math, float32, in the reference's operation order ---------------------------

// MuZeroNet._signed_parabolic (networks.py:186-189) applied to the support expectation x:
//   z = sqrt(1 + 4*eps*(eps + 1 + |x|)) / 2 / eps - 1/2/eps ;  sign(x) * (z*z - 1),  eps = 1e-3
// with python scalars folded the way torch folds them (4*eps = 0.004, eps+1 = 1.001,
// 1/2/eps = 500.0, each rounded to float32 when it meets the tensor).
__device__ __forceinline__ float signed_parabolic(float x) {
  const float a = __fadd_rn(1.001f, fabsf(x));
  const float s = __fsqrt_rn(__fadd_rn(1.0f, __fmul_rn(0.004f, a)));
  const float z = __fsub_rn(__fdiv_rn(__fdiv_rn(s, 2.0f), 0.001f), 500.0f);
  const float sg = (x > 0.0f) ? 1.0f : ((x < 0.0f) ? -1.0f : 0.0f);
  return __fmul_rn(sg, __fsub_rn(__fmul_rn(z, z), 1.0f));
}

// logits_to_transformed_expected_value (networks.py:152-184): softmax over the 33 support
// logits, expectation over linspace(-16, 16, 33), then the signed-parabolic transform.
// `get(i)` returns logit i.
template <typename F>
__device__ __forceinline__ float support_to_scalar(F get) {
  float mx = get(0);
#pragma unroll
  for (int i = 1; i < kSupport; ++i) mx = fmaxf(mx, get(i));
  float den = 0.0f, num = 0.0f;
#pragma unroll
  for (int i = 0; i < kSupport; ++i) {
    const float e = expf(get(i) - mx);
    den += e;
    num = fmaf(e, (float)(i - (kSupport - 1) / 2), num);
  }
  return signed_parabolic(__fdiv_rn(num, den));
}

}  // namespace hmz
