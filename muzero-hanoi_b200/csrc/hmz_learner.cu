// The learner step (SURVEY.md §8f row 4): Muzero._update (reference Muzero.py:209-274) + MuZeroNet.update
// (networks.py:118-122, Adam of networks.py:69) for one batch, forward and backward written out by hand.
//
//   h_0 = normalize(representation_net(s));  for t in 0..K-1:
//     pi_t = policy_net(h_t);  v_t = T(value_net(h_t));  x = dynamic_net([h_t, onehot(a_t)]);
//     r_t = T(rwd_net(x));  h_{t+1} = normalize(x) with its incoming gradient halved (Muzero.py:235)
//   loss_b = sum_t (v_t - G_t)^2 + (r_t - R_t)^2 + CE(pi_t, pi*_t);  L = mean_b(w_b loss_b), gradient x 1/K (:264)
// T = softmax expectation over the 33-bin support + signed parabolic (networks.py:152-189).
//
// Everything is float32 like the reference (torch CPU float32); sums run in a different order than torch's
// BLAS, so parity is to ~1e-5 relative on gradients, not bit-exact.  The batch is small (256 x 5 unroll steps,
// ~1 GFLOP per update): these are plain tiled FFMA kernels, one launch per layer — the acting path is where
// the tensor cores are; nothing here is on it.
#include <cmath>
#include <vector>

#include "hmz_net.cuh"

namespace hmz {
namespace learner {

constexpr int kTile = 32;

// Y[M,N] = X[M,K] W[N,K]^T + b  (optionally relu)
__global__ void __launch_bounds__(256) lin_fwd(const float* __restrict__ X, int ldx, const float* __restrict__ W, const float* __restrict__ b,
                                               float* __restrict__ Y, int ldy, int M, int N, int K, int relu) {
  __shared__ float xs[kTile][kTile + 1], ws[kTile][kTile + 1];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8 threads, 4 rows each
  const int m0 = blockIdx.y * kTile, n0 = blockIdx.x * kTile;
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
  for (int k0 = 0; k0 < K; k0 += kTile) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int r = ty * 4 + i;
      xs[r][tx] = (m0 + r < M && k0 + tx < K) ? X[(size_t)(m0 + r) * ldx + k0 + tx] : 0.f;
      ws[r][tx] = (n0 + r < N && k0 + tx < K) ? W[(size_t)(n0 + r) * K + k0 + tx] : 0.f;
    }
    __syncthreads();
#pragma unroll 8
    for (int k = 0; k < kTile; ++k) {
      const float w = ws[tx][k];
#pragma unroll
      for (int i = 0; i < 4; ++i) acc[i] = fmaf(xs[ty * 4 + i][k], w, acc[i]);
    }
    __syncthreads();
  }
  if (n0 + tx < N) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int m = m0 + ty * 4 + i;
      if (m < M) {
        float y = acc[i] + b[n0 + tx];
        if (relu) y = fmaxf(y, 0.f);
        Y[(size_t)m * ldy + n0 + tx] = y;
      }
    }
  }
}

// dX[M,K] (+)= dY[M,N] W[N,K]   (accumulate != 0 adds to dX)
__global__ void __launch_bounds__(256) lin_bwd_dx(const float* __restrict__ dY, int ldy, const float* __restrict__ W, float* __restrict__ dX,
                                                  int ldx, int M, int N, int K, int k_out, int accumulate) {
  __shared__ float ys[kTile][kTile + 1], ws[kTile][kTile + 1];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int m0 = blockIdx.y * kTile, k0 = blockIdx.x * kTile;
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
  for (int n0 = 0; n0 < N; n0 += kTile) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int r = ty * 4 + i;
      ys[r][tx] = (m0 + r < M && n0 + tx < N) ? dY[(size_t)(m0 + r) * ldy + n0 + tx] : 0.f;
      ws[r][tx] = (n0 + r < N && k0 + tx < K) ? W[(size_t)(n0 + r) * K + k0 + tx] : 0.f;  // ws[n][k]
    }
    __syncthreads();
#pragma unroll 8
    for (int n = 0; n < kTile; ++n) {
      const float w = ws[n][tx];
#pragma unroll
      for (int i = 0; i < 4; ++i) acc[i] = fmaf(ys[ty * 4 + i][n], w, acc[i]);
    }
    __syncthreads();
  }
  if (k0 + tx < k_out) {  // k_out <= K: the one-hot action columns of dynamic_net.0 get no gradient consumer
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int m = m0 + ty * 4 + i;
      if (m < M) {
        float* p = dX + (size_t)m * ldx + k0 + tx;
        *p = accumulate ? *p + acc[i] : acc[i];
      }
    }
  }
}

// dW[N,K] += dY[M,N]^T X[M,K];  db[N] += sum_m dY[m,n]   (gradients accumulate over the unroll steps).
// Each 32-row tile is summed on its own and then added to the running sum, so float32 rounding grows with
// 32 + M / 32 additions instead of M (the batch is 4,096 rows in the tests).
__global__ void __launch_bounds__(256) lin_bwd_dw(const float* __restrict__ dY, int ldy, const float* __restrict__ X, int ldx,
                                                  float* __restrict__ dW, float* __restrict__ db, int M, int N, int K) {
  __shared__ float ys[kTile][kTile + 1], xs[kTile][kTile + 1];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int n0 = blockIdx.y * kTile, k0 = blockIdx.x * kTile;
  float acc[4] = {0.f, 0.f, 0.f, 0.f}, bsum[4] = {0.f, 0.f, 0.f, 0.f};
  for (int m0 = 0; m0 < M; m0 += kTile) {
    float part[4] = {0.f, 0.f, 0.f, 0.f}, bpart[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int r = ty * 4 + i;  // r = m inside the tile
      ys[r][tx] = (m0 + r < M && n0 + tx < N) ? dY[(size_t)(m0 + r) * ldy + n0 + tx] : 0.f;  // ys[m][n]
      xs[r][tx] = (m0 + r < M && k0 + tx < K) ? X[(size_t)(m0 + r) * ldx + k0 + tx] : 0.f;   // xs[m][k]
    }
    __syncthreads();
#pragma unroll 8
    for (int m = 0; m < kTile; ++m) {
      const float x = xs[m][tx];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float y = ys[m][ty * 4 + i];
        part[i] = fmaf(y, x, part[i]);
        if (blockIdx.x == 0 && tx == 0) bpart[i] += y;
      }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      acc[i] += part[i];
      bsum[i] += bpart[i];
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int n = n0 + ty * 4 + i;
    if (n < N) {
      if (k0 + tx < K) dW[(size_t)n * K + k0 + tx] += acc[i];
      if (blockIdx.x == 0 && tx == 0) db[n] += bsum[i];
    }
  }
}

// dH *= (H > 0)
__global__ void __launch_bounds__(256) relu_bwd(float* __restrict__ dH, const float* __restrict__ H, int64_t n) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    if (!(H[i] > 0.f)) dH[i] = 0.f;
}

// X[b] = [h[b, 0:64], onehot(action[b, t])]   (torch.cat, networks.py:130)
__global__ void __launch_bounds__(256) concat_action(const float* __restrict__ h, const int64_t* __restrict__ actions, int t, int unroll,
                                                     float* __restrict__ X, int B) {
  const int width = kLatent + kActions;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < B * width; i += gridDim.x * blockDim.x) {
    const int b = i / width, c = i - b * width;
    X[i] = c < kLatent ? h[b * kLatent + c] : ((int64_t)(c - kLatent) == actions[(size_t)b * unroll + t] ? 1.f : 0.f);
  }
}

// normalize_h_state (networks.py:191-196): y = (h - min) / (max - min + 1e-8); keeps argmin / argmax (first
// occurrence, as torch.min / torch.max over a dim return) for the backward pass.
__global__ void __launch_bounds__(256) normalize_fwd(const float* __restrict__ h, float* __restrict__ y, int32_t* __restrict__ arg, int B) {
  for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < B; b += gridDim.x * blockDim.x) {
    const float* r = h + (size_t)b * kLatent;
    float mn = r[0], mx = r[0];
    int imn = 0, imx = 0;
    for (int i = 1; i < kLatent; ++i) {
      if (r[i] < mn) { mn = r[i]; imn = i; }
      if (r[i] > mx) { mx = r[i]; imx = i; }
    }
    const float D = (mx - mn) + 1e-8f;
    for (int i = 0; i < kLatent; ++i) y[(size_t)b * kLatent + i] = (r[i] - mn) / D;
    arg[2 * b] = imn;
    arg[2 * b + 1] = imx;
  }
}
// dh = scale * g / D everywhere, plus the gradients routed through min and max to their arg indices;
// added to dh (which may already hold the reward head's gradient on the raw latent) when accumulate != 0.
__global__ void __launch_bounds__(256) normalize_bwd(const float* __restrict__ g, float scale, const float* __restrict__ h,
                                                     const int32_t* __restrict__ arg, float* __restrict__ dh, int B, int accumulate) {
  for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < B; b += gridDim.x * blockDim.x) {
    const float* r = h + (size_t)b * kLatent;
    const int imn = arg[2 * b], imx = arg[2 * b + 1];
    const float mn = r[imn], D = (r[imx] - mn) + 1e-8f;
    float dmin = 0.f, dmax = 0.f;
    for (int i = 0; i < kLatent; ++i) {
      const float gi = g[(size_t)b * kLatent + i] * scale;
      const float u = (r[i] - mn) / (D * D);
      dmin += gi * (u - 1.f / D);
      dmax -= gi * u;
      float* p = dh + (size_t)b * kLatent + i;
      *p = (accumulate ? *p : 0.f) + gi / D;
    }
    dh[(size_t)b * kLatent + imn] += dmin;
    dh[(size_t)b * kLatent + imx] += dmax;
  }
}

// logits_to_transformed_expected_value (networks.py:152-189) + squared-error loss against `target`:
//   out = T(logits);  loss_b += (out - target)^2;  dlogits = coef_b * 2 (out - target) * dT/dlogits
// first_pred (nullable): |out - target| of unroll step 0 = the new priorities (Muzero.py:253-258).
__global__ void __launch_bounds__(128) support_loss(const float* __restrict__ logits, const float* __restrict__ target, int t, int unroll,
                                                    const float* __restrict__ coef, float* __restrict__ dlogits,
                                                    double* __restrict__ loss_acc, float* __restrict__ first_pred, int B) {
  for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < B; b += gridDim.x * blockDim.x) {
    const float* l = logits + (size_t)b * kSupport;
    float mx = l[0];
    for (int i = 1; i < kSupport; ++i) mx = fmaxf(mx, l[i]);
    // x = sum_i e_i (i - 16) / sum_i e_i over the unnormalised exponentials, as support_to_scalar (hmz_net.cuh) forms
    // it: all-equal logits give e_i = 1 and x = 0 exactly (as torch's float32 sum(softmax * linspace) does), so that
    // row's sign(x) is 0 and it sends no gradient.  Normalising first would leave x a few ulps off 0 with sign -1.
    float p[kSupport], den = 0.f, num = 0.f;
    for (int i = 0; i < kSupport; ++i) {
      p[i] = expf(l[i] - mx);
      den += p[i];
      num = fmaf(p[i], (float)(i - (kSupport - 1) / 2), num);
    }
    const float x = __fdiv_rn(num, den);
    for (int i = 0; i < kSupport; ++i) p[i] /= den;
    // MuZeroNet._signed_parabolic in the reference's float32 operation order (see signed_parabolic, hmz_net.cuh)
    const float root = __fsqrt_rn(__fadd_rn(1.0f, __fmul_rn(0.004f, __fadd_rn(1.001f, fabsf(x)))));
    const float z = __fsub_rn(__fdiv_rn(__fdiv_rn(root, 2.0f), 0.001f), 500.0f);
    const float sg = x > 0.f ? 1.f : (x < 0.f ? -1.f : 0.f);
    const float out = __fmul_rn(sg, __fsub_rn(__fmul_rn(z, z), 1.0f));
    const float diff = out - target[(size_t)b * unroll + t];
    atomicAdd(loss_acc, (double)(diff * diff));
    if (first_pred && t == 0) first_pred[b] = fabsf(diff);
    // d out / d x = sign(x)^2 * 2 z / root  (0 at x == 0, where torch.sign has value and gradient 0)
    const float gx = coef[b] * 2.f * diff * (sg * sg) * 2.f * z / root;
    for (int i = 0; i < kSupport; ++i) dlogits[(size_t)b * kSupport + i] = gx * p[i] * ((float)(i - (kSupport - 1) / 2) - x);
  }
}

// F.cross_entropy(logits, soft target, reduction="none") (Muzero.py:243-245):
//   loss_b += -sum_k t_k log_softmax(l)_k;  dlogits = coef_b (softmax(l) sum_k t_k - t)
__global__ void __launch_bounds__(128) policy_loss(const float* __restrict__ logits, const float* __restrict__ pi_target, int t, int unroll,
                                                   const float* __restrict__ coef, float* __restrict__ dlogits,
                                                   double* __restrict__ loss_acc, int B) {
  for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < B; b += gridDim.x * blockDim.x) {
    const float* l = logits + (size_t)b * kActions;
    const float* tg = pi_target + ((size_t)b * unroll + t) * kActions;
    float mx = l[0];
    for (int i = 1; i < kActions; ++i) mx = fmaxf(mx, l[i]);
    float den = 0.f, tsum = 0.f;
    for (int i = 0; i < kActions; ++i) {
      den += expf(l[i] - mx);
      tsum += tg[i];
    }
    const float lse = logf(den) + mx;
    float loss = 0.f;
    for (int i = 0; i < kActions; ++i) {
      loss -= tg[i] * (l[i] - lse);
      dlogits[(size_t)b * kActions + i] = coef[b] * (expf(l[i] - lse) * tsum - tg[i]);
    }
    atomicAdd(loss_acc, (double)loss);
  }
}

// coef_b = w_b / (B K): loss * priority_w, .mean(), gradient x 1 / unroll (Muzero.py:250,260,264)
__global__ void __launch_bounds__(256) make_coef(const float* __restrict__ w, float* __restrict__ coef, int B, int unroll) {
  for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < B; b += gridDim.x * blockDim.x)
    coef[b] = (w ? w[b] : 1.f) / ((float)B * (float)unroll);
}

// torch.optim.Adam (default betas / eps, no weight decay, networks.py:69), single-tensor form:
//   exp_avg.lerp_(grad, 1 - beta1);  exp_avg_sq.mul_(beta2).addcmul_(grad, grad, value=1 - beta2);
//   denom = exp_avg_sq.sqrt() / sqrt(bias2) + eps;  param.addcdiv_(exp_avg, denom, value=-lr / bias1)
// Every scalar is a double on the host (1 - beta1 in double, not 1 - (float)beta1) rounded once to float32 here.
__global__ void __launch_bounds__(256) adam_step(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                                 float* __restrict__ v, int64_t n, float one_m_beta1, float beta2, float one_m_beta2,
                                                 float eps, float bias2_sqrt, float neg_step) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float gi = g[i];
    const float mi = m[i] + one_m_beta1 * (gi - m[i]);
    const float vi = v[i] * beta2 + one_m_beta2 * gi * gi;
    m[i] = mi;
    v[i] = vi;
    const float denom = sqrtf(vi) / bias2_sqrt + eps;
    p[i] += neg_step * (mi / denom);
  }
}

__global__ void __launch_bounds__(256) zero_f32(float* __restrict__ p, int64_t n) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) p[i] = 0.f;
}
__global__ void zero_f64(double* __restrict__ p, int n) {
  if ((int)threadIdx.x < n) p[threadIdx.x] = 0.0;
}
// losses_out = the double sums / B, rounded once
__global__ void scale_losses(const double* __restrict__ sums, float* __restrict__ losses_out, double inv_b) {
  if (threadIdx.x < 3) losses_out[threadIdx.x] = (float)(sums[threadIdx.x] * inv_b);
}

// ---- flat parameter layout: the 20 tensors of MuZeroNet.state_dict() in state_dict order, torch [out][in] ----
struct Mlp {
  int w1, b1, w2, b2;  // offsets (floats)
  int in, out;
};
struct Layout {
  Mlp rep, dyn, rwd, pol, val;
  int total;
};
static Layout make_layout(int n_disks) {
  Layout L;
  int at = 0;
  auto mlp = [&](int in, int out) {
    Mlp m;
    m.in = in;
    m.out = out;
    m.w1 = at; at += kHidden * in;
    m.b1 = at; at += kHidden;
    m.w2 = at; at += out * kHidden;
    m.b2 = at; at += out;
    return m;
  };
  L.rep = mlp(3 * n_disks, kLatent);
  L.dyn = mlp(kLatent + kActions, kLatent);
  L.rwd = mlp(kLatent, kSupport);
  L.pol = mlp(kLatent, kActions);
  L.val = mlp(kLatent, kSupport);
  L.total = at;
  return L;
}

// per unroll step activations (floats per batch row)
struct StepBuf {
  float *h, *x, *hid_dyn, *h_raw, *hid_rwd, *r_logits, *hid_pol, *pi_logits, *hid_val, *v_logits;
  int32_t* arg;  // argmin / argmax of h_raw
};
constexpr int kStepFloats = kLatent + (kLatent + kActions) + kHidden + kLatent + kHidden + kSupport + kHidden + kActions + kHidden + kSupport + 2;

static inline dim3 gemm_grid(int cols, int rows) { return dim3((cols + kTile - 1) / kTile, (rows + kTile - 1) / kTile); }

}  // namespace learner
}  // namespace hmz

using namespace hmz;
using namespace hmz::learner;

extern "C" {

int64_t hmz_learner_param_count(int n_disks) {
  if (n_disks < 1 || n_disks > HMZ_MAX_DISKS) return -1;
  return make_layout(n_disks).total;
}

int64_t hmz_learner_workspace_bytes(int n_disks, int batch, int unroll) {
  if (n_disks < 1 || n_disks > HMZ_MAX_DISKS || batch < 1 || unroll < 1) return -1;
  // rep activations + (unroll + 1) latents + per-step buffers + gradient scratch
  const int64_t per_row = (int64_t)kHidden + kLatent + 2 + (int64_t)unroll * kStepFloats + kLatent /* h_K */ +
                          /* scratch: */ 2 * kLatent + (kLatent + kActions) + 2 * kHidden + 2 * kSupport + kActions + 1 /* coef */;
  return (per_row * batch + 16) * 4 + 256;
}

int hmz_learner_step(float* params, float* grads, float* adam_m, float* adam_v, void* workspace, int n_disks, int batch, int unroll,
                     const float* states, const float* rwds, const int64_t* actions, const float* pi_probs, const float* returns,
                     const float* priority_w, double lr, double beta1, double beta2, double eps, int64_t step_index,
                     float* new_priorities, float* losses_out, int apply_update, void* stream) {
  ProfScope prof_scope(HMZ_PROF_OTHER, stream);
  if (!params || !grads || !workspace || !states || !rwds || !actions || !pi_probs || !returns || !losses_out || batch < 1 ||
      unroll < 1 || n_disks < 1 || n_disks > HMZ_MAX_DISKS || step_index < 1 || (apply_update && (!adam_m || !adam_v)))
    return fail(HMZ_ERR_INVALID, "hmz_learner_step: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  const Layout L = make_layout(n_disks);
  const int B = batch, K = unroll, d_in = 3 * n_disks;
  float* ws = (float*)(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
  auto take = [&](int64_t per_row) {
    float* p = ws;
    ws += per_row * B;
    return p;
  };
  float* hid_rep = take(kHidden);
  float* h_raw0 = take(kLatent);
  int32_t* arg0 = (int32_t*)take(2);
  std::vector<StepBuf> sb(K);
  float* h0 = take(kLatent);
  float* h_cur = h0;
  for (int t = 0; t < K; ++t) {
    StepBuf& s = sb[t];
    s.h = h_cur;
    s.x = take(kLatent + kActions);
    s.hid_dyn = take(kHidden);
    s.h_raw = take(kLatent);
    s.hid_rwd = take(kHidden);
    s.r_logits = take(kSupport);
    s.hid_pol = take(kHidden);
    s.pi_logits = take(kActions);
    s.hid_val = take(kHidden);
    s.v_logits = take(kSupport);
    s.arg = (int32_t*)take(2);
    h_cur = take(kLatent);  // h_{t+1}
  }
  float* g_h = take(kLatent);       // gradient w.r.t. the normalised latent of the current step
  float* g_hraw = take(kLatent);    // gradient w.r.t. a raw (pre-normalisation) latent
  float* g_x = take(kLatent + kActions);
  float* g_hid = take(kHidden);
  float* g_hid2 = take(kHidden);
  float* g_l33 = take(kSupport);
  float* g_l33b = take(kSupport);
  float* g_l6 = take(kActions);
  float* coef = take(1);
  double* loss3 = (double*)(((uintptr_t)ws + 7) & ~(uintptr_t)7);  // value, reward, policy loss sums (in the 64-byte tail)

  auto fwd = [&](const float* X, int ldx, const float* W, const float* b, float* Y, int ldy, int N, int Kd, int relu) {
    lin_fwd<<<gemm_grid(N, B), 256, 0, st>>>(X, ldx, W, b, Y, ldy, B, N, Kd, relu);
    g_launches.fetch_add(1, std::memory_order_relaxed);
  };
  auto mlp_fwd = [&](const Mlp& m, const float* X, float* hid, float* out) {
    fwd(X, m.in, params + m.w1, params + m.b1, hid, kHidden, kHidden, m.in, 1);
    fwd(hid, kHidden, params + m.w2, params + m.b2, out, m.out, m.out, kHidden, 0);
  };
  // backward of an MLP given d(out) in g_out: accumulates dW / db, leaves d(in) in g_in (first k_out columns)
  auto mlp_bwd = [&](const Mlp& m, const float* X, const float* hid, const float* g_out, float* g_hidden, float* g_in, int k_out,
                     int accumulate_in) {
    lin_bwd_dw<<<gemm_grid(kHidden, m.out), 256, 0, st>>>(g_out, m.out, hid, kHidden, grads + m.w2, grads + m.b2, B, m.out, kHidden);
    lin_bwd_dx<<<gemm_grid(kHidden, B), 256, 0, st>>>(g_out, m.out, params + m.w2, g_hidden, kHidden, B, m.out, kHidden, kHidden, 0);
    relu_bwd<<<grid_for((int64_t)B * kHidden, 256, 4), 256, 0, st>>>(g_hidden, hid, (int64_t)B * kHidden);
    lin_bwd_dw<<<gemm_grid(m.in, kHidden), 256, 0, st>>>(g_hidden, kHidden, X, m.in, grads + m.w1, grads + m.b1, B, kHidden, m.in);
    if (g_in)
      lin_bwd_dx<<<gemm_grid(k_out, B), 256, 0, st>>>(g_hidden, kHidden, params + m.w1, g_in, k_out == m.in ? m.in : k_out, B, kHidden, m.in,
                                                      k_out, accumulate_in);
    g_launches.fetch_add(g_in ? 5 : 4, std::memory_order_relaxed);
  };

  zero_f32<<<grid_for(L.total, 256, 8), 256, 0, st>>>(grads, L.total);
  zero_f64<<<1, 32, 0, st>>>(loss3, 3);
  make_coef<<<grid_for(B, 256, 1), 256, 0, st>>>(priority_w, coef, B, K);
  // ---- forward
  mlp_fwd(L.rep, states, hid_rep, h_raw0);
  normalize_fwd<<<grid_for(B, 256, 1), 256, 0, st>>>(h_raw0, h0, arg0, B);
  for (int t = 0; t < K; ++t) {
    StepBuf& s = sb[t];
    mlp_fwd(L.pol, s.h, s.hid_pol, s.pi_logits);
    mlp_fwd(L.val, s.h, s.hid_val, s.v_logits);
    concat_action<<<grid_for((int64_t)B * (kLatent + kActions), 256, 2), 256, 0, st>>>(s.h, actions, t, K, s.x, B);
    mlp_fwd(L.dyn, s.x, s.hid_dyn, s.h_raw);
    mlp_fwd(L.rwd, s.h_raw, s.hid_rwd, s.r_logits);
    float* h_next = (t + 1 < K) ? sb[t + 1].h : h_cur;
    normalize_fwd<<<grid_for(B, 256, 1), 256, 0, st>>>(s.h_raw, h_next, s.arg, B);
  }
  // ---- backward, last unroll step first
  for (int t = K - 1; t >= 0; --t) {
    StepBuf& s = sb[t];
    // reward head on the raw new latent: d h_raw
    support_loss<<<grid_for(B, 128, 1), 128, 0, st>>>(s.r_logits, rwds, t, K, coef, g_l33, loss3 + 1, nullptr, B);
    mlp_bwd(L.rwd, s.h_raw, s.hid_rwd, g_l33, g_hid, g_hraw, kLatent, 0);
    // gradient arriving at h_{t+1} from the later steps, halved by the hook of Muzero.py:235, through the normalisation
    if (t + 1 < K) normalize_bwd<<<grid_for(B, 256, 1), 256, 0, st>>>(g_h, 0.5f, s.h_raw, s.arg, g_hraw, B, 1);
    // dynamics: d [h_t, onehot] -> g_h (the first 64 columns)
    mlp_bwd(L.dyn, s.x, s.hid_dyn, g_hraw, g_hid, g_h, kLatent, 0);
    // prediction heads on h_t
    policy_loss<<<grid_for(B, 128, 1), 128, 0, st>>>(s.pi_logits, pi_probs, t, K, coef, g_l6, loss3 + 2, B);
    mlp_bwd(L.pol, s.h, s.hid_pol, g_l6, g_hid2, g_h, kLatent, 1);
    support_loss<<<grid_for(B, 128, 1), 128, 0, st>>>(s.v_logits, returns, t, K, coef, g_l33b, loss3 + 0, new_priorities, B);
    mlp_bwd(L.val, s.h, s.hid_val, g_l33b, g_hid2, g_h, kLatent, 1);
  }
  // representation: h_0 has no hook
  normalize_bwd<<<grid_for(B, 256, 1), 256, 0, st>>>(g_h, 1.0f, h_raw0, arg0, g_hraw, B, 0);
  mlp_bwd(L.rep, states, hid_rep, g_hraw, g_hid, nullptr, d_in, 0);
  scale_losses<<<1, 32, 0, st>>>(loss3, losses_out, 1.0 / (double)B);
  if (apply_update) {
    // torch evaluates the bias corrections and the step size in double on the host
    const double bias1 = 1.0 - std::pow(beta1, (double)step_index), bias2 = 1.0 - std::pow(beta2, (double)step_index);
    adam_step<<<grid_for(L.total, 256, 8), 256, 0, st>>>(params, grads, adam_m, adam_v, L.total, (float)(1.0 - beta1), (float)beta2,
                                                         (float)(1.0 - beta2), (float)eps, (float)std::sqrt(bias2), (float)(-lr / bias1));
  }
  (void)g_x;
  return check_launch("hmz_learner_step");
}

}  // extern "C"
