// Prioritized replay sampling on the device: ReplayRing.priority_sample (buffer.py:96 of the reference) and
// update_priorities (:130), bit-exact with NumPy, so that a learner update needs no host round trip.
//
// The chain NumPy runs (priority exponent 1, float32 priorities q of the num filled rows):
//   s   = np.sum(q)                 float32, NumPy's pairwise tree (replay_sum_leaves + the top of replay_draw)
//   x   = q / s                     float32, one IEEE division per row
//   np.random.choice(num, batch, p=x): p = float64(x); Kahan-sum / sign checks; cdf = cumsum(p) strictly left to right;
//       cdf /= cdf[-1]; idx = searchsorted(cdf, u, side="right") for the caller's uniforms u
//   w   = (float32(1 / size) / x[idx]) ** beta;  w /= max(w)
//
// The cumulative sum is the only sequential step.  It is evaluated exactly in parallel, stretch by stretch: while the
// running sum c stays in one binade [2^e, 2^(e+1)) it is a multiple of u = 2^(e-52), and c + x rounds to
// c + u * (floor(x/u) + r), where r depends on x alone (remainder below / above u/2) except at an exact half, where
// ties-to-even makes r the parity of c/u + floor(x/u).  Each row is therefore a map from the incoming parity bit to
// (increment, outgoing parity bit); these maps compose associatively, so a block scan yields every c of the stretch.
// A stretch ends at the first row whose sum reaches 2^(e+1): that row is added with an ordinary double add and the next
// stretch starts in the new binade.  Leading zero rows leave c at 0 until the first non-zero row, which sets c exactly.
// c only grows, so a ring has at most a few dozen stretches.  One CTA walks the ring in chunks of 8,192 rows; a chunk
// in which a stretch ends is resumed after that row.
#include <climits>

#include "hmz_common.cuh"

namespace hmz {
namespace {

constexpr int kLeaf = 128;       // NumPy adds blocks of <= 128 elements with eight accumulators (PW_BLOCKSIZE)
constexpr int kSumThreads = 256; // virtual-tree positions per CTA of replay_sum_leaves: its bottom 8 levels
constexpr int kTopBits = 13;     // replay_draw reduces at most 2^13 partial sums in shared memory
constexpr int kDrawThreads = 1024;
constexpr int kItems = 8;
constexpr int kChunk = kDrawThreads * kItems;
constexpr unsigned long long kTop = 1ull << 53;  // c / u reaches 2^53: the stretch's binade is left
constexpr unsigned long long kSat = 1ull << 54;  // increments saturate here (any value >= 2^53 ends the stretch)
// |kahan_sum(p) - 1| > atol with atol = float32(sqrt(float32 eps)) (numpy/random/mtrand.pyx, RandomState.choice)
constexpr double kSumAtol = 0x1.6a09e6p-12;

// Depth of NumPy's pairwise tree over n elements: a node of more than 128 elements splits at n/2 rounded down to a
// multiple of 8; the right part is the larger, so it is the deepest.
int pairwise_depth(int64_t n) {
  int d = 0;
  while (n > kLeaf) {
    n -= (n / 2) & ~(int64_t)7;
    ++d;
  }
  return d;
}

// One leaf of NumPy's pairwise_sum (numpy/_core/src/umath/loops_utils.h.src), float32 with round-to-nearest adds.
__device__ float pairwise_leaf(const float* __restrict__ a, int n) {
  if (n < 8) {
    float res = -0.0f;
    for (int i = 0; i < n; ++i) res = __fadd_rn(res, a[i]);
    return res;
  }
  float r[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) r[j] = a[j];
  int i = 8;
  for (; i < n - (n % 8); i += 8) {
#pragma unroll
    for (int j = 0; j < 8; ++j) r[j] = __fadd_rn(r[j], a[i + j]);
  }
  float res = __fadd_rn(__fadd_rn(__fadd_rn(r[0], r[1]), __fadd_rn(r[2], r[3])), __fadd_rn(__fadd_rn(r[4], r[5]), __fadd_rn(r[6], r[7])));
  for (; i < n; ++i) res = __fadd_rn(res, a[i]);
  return res;
}

// The pairwise tree laid out as a complete binary tree of depth `depth` (>= 8): position t's path from the root is its
// bits, most significant first.  The walk stops at the first node of <= 128 elements (a leaf); position t holds that
// leaf if the remaining bits are zero.  A node of the complete tree "exists" if it is a real node or the leftmost
// descendant of a leaf; then a parent's value is left + right when its right child exists and left's value otherwise,
// which reproduces the real tree exactly.  Each CTA reduces the bottom 8 levels of its 256 positions.
__global__ void __launch_bounds__(kSumThreads) replay_sum_leaves(const float* __restrict__ q, int64_t num, int depth,
                                                                 float* __restrict__ part, uint8_t* __restrict__ part_exists) {
  __shared__ float v[kSumThreads];
  __shared__ uint8_t ex[kSumThreads];
  const int64_t t = (int64_t)blockIdx.x * kSumThreads + threadIdx.x;
  int64_t a = 0, n = num;
  int l = 0;
  for (; l < depth && n > kLeaf; ++l) {
    const int64_t m = (n / 2) & ~(int64_t)7;
    if ((t >> (depth - 1 - l)) & 1) {
      a += m;
      n -= m;
    } else {
      n = m;
    }
  }
  const bool owner = (t & ((1ll << (depth - l)) - 1)) == 0;
  v[threadIdx.x] = owner ? pairwise_leaf(q + a, (int)n) : 0.0f;
  ex[threadIdx.x] = owner;
  __syncthreads();
  for (int w = kSumThreads / 2; w >= 1; w >>= 1) {
    float r = 0.0f;
    uint8_t e = 0;
    if (threadIdx.x < w) {
      const int k = threadIdx.x;
      e = ex[2 * k];
      r = ex[2 * k + 1] ? __fadd_rn(v[2 * k], v[2 * k + 1]) : v[2 * k];
    }
    __syncthreads();
    if (threadIdx.x < w) {
      v[threadIdx.x] = r;
      ex[threadIdx.x] = e;
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    part[blockIdx.x] = v[0];
    part_exists[blockIdx.x] = ex[0];
  }
}

// Row map of the exact cumulative sum: for incoming parity bit b of c/u, c/u grows by inc[b] and leaves with parity
// bit (bits >> b) & 1.
struct RowMap {
  unsigned long long inc0, inc1;
  unsigned bits;
};

__device__ __forceinline__ RowMap identity_map() { return RowMap{0ull, 0ull, 2u}; }

__device__ __forceinline__ unsigned long long sat_add(unsigned long long a, unsigned long long b) {
  const unsigned long long s = a + b;  // both <= 2^54: no overflow
  return s < kSat ? s : kSat;
}

// f, then g
__device__ __forceinline__ RowMap compose(const RowMap& f, const RowMap& g) {
  const unsigned f0 = f.bits & 1u, f1 = (f.bits >> 1) & 1u;
  RowMap h;
  h.inc0 = sat_add(f.inc0, f0 ? g.inc1 : g.inc0);
  h.inc1 = sat_add(f.inc1, f1 ? g.inc1 : g.inc0);
  h.bits = ((g.bits >> f0) & 1u) | (((g.bits >> f1) & 1u) << 1);
  return h;
}

// x (a float32 value widened, >= 0) added to a running sum whose binade has biased exponent E: x / u = n + remainder,
// cls = 0 for a remainder below one half, 1 above, 2 exactly one half (the tie).  n saturates at 2^54.
__device__ __forceinline__ void row_parts(double x, int E, unsigned long long& n, int& cls) {
  cls = 0;
  if (!(x > 0.0)) {
    n = 0;
    return;
  }
  const unsigned long long xb = (unsigned long long)__double_as_longlong(x);
  const int sh = (int)(xb >> 52) - E;  // x / u = mx * 2^sh
  const unsigned long long mx = (xb & ((1ull << 52) - 1)) | (1ull << 52);
  if (sh > 0) {
    n = kSat;
  } else if (sh == 0) {
    n = mx;
  } else if (sh < -60) {
    n = 0;  // x < u / 2^7
  } else {
    const int k = -sh;
    n = mx >> k;
    const unsigned long long rem = mx & ((1ull << k) - 1), half = 1ull << (k - 1);
    cls = rem > half ? 1 : (rem == half ? 2 : 0);
  }
}

// c / u after adding the row to c / u = v (< 2^53): ties go to the even result
__device__ __forceinline__ unsigned long long row_add(unsigned long long v, unsigned long long n, int cls) {
  return v + (cls == 2 ? n + ((v + n) & 1ull) : sat_add(n, (unsigned long long)cls));
}

__device__ __forceinline__ RowMap row_map(double x, int E) {
  unsigned long long n;
  int cls;
  row_parts(x, E, n, cls);
  RowMap m;
  if (cls != 2) {
    const unsigned long long inc = sat_add(n, (unsigned long long)cls);
    const unsigned p = (unsigned)(inc & 1ull);
    m.inc0 = m.inc1 = inc;
    m.bits = p | ((p ^ 1u) << 1);
  } else {  // ties to even: the result c/u + n + r is even
    m.inc0 = n + (n & 1ull);
    m.inc1 = n + ((n & 1ull) ^ 1ull);
    m.bits = 0u;
  }
  return m;
}

// c = (mantissa with hidden bit) * u in the binade of biased exponent E; val in [2^52, 2^53] (2^53 = the next binade)
__device__ __forceinline__ double make_c(int E, unsigned long long val) {
  return __longlong_as_double((long long)(((unsigned long long)E << 52) + val - (1ull << 52)));
}

__device__ __forceinline__ RowMap shfl_up_map(const RowMap& m, int d) {
  RowMap r;
  r.inc0 = __shfl_up_sync(0xffffffffu, m.inc0, d);
  r.inc1 = __shfl_up_sync(0xffffffffu, m.inc1, d);
  r.bits = __shfl_up_sync(0xffffffffu, m.bits, d);
  return r;
}

// NaN-propagating max (np.max)
__device__ __forceinline__ float nan_max(float a, float b) { return (a != a || b != b) ? __int_as_float(0x7fc00000) : fmaxf(a, b); }

__device__ __forceinline__ int block_min(int v, int* red) {
  v = __reduce_min_sync(0xffffffffu, v);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  if (threadIdx.x < 32) {
    int w = red[threadIdx.x];
    w = __reduce_min_sync(0xffffffffu, w);
    if (threadIdx.x == 0) red[32] = w;
  }
  __syncthreads();
  const int r = red[32];
  __syncthreads();
  return r;
}

// The top of the pairwise sum, the division, NumPy's checks, the exact cumulative sum, the search and the weights.
__global__ void __launch_bounds__(kDrawThreads) replay_draw(const float* __restrict__ q, int64_t num, int top_levels,
                                                            const float* __restrict__ part, const uint8_t* __restrict__ part_exists,
                                                            double* __restrict__ cdf, const double* __restrict__ uniforms, int64_t batch,
                                                            float inv_size, float beta, int64_t* __restrict__ indices,
                                                            float* __restrict__ weights, int32_t* __restrict__ status) {
  __shared__ float tv[1 << kTopBits];
  __shared__ uint8_t te[1 << kTopBits];
  __shared__ RowMap warp_maps[32];
  __shared__ unsigned long long warp_incs[32];
  __shared__ int red[33];
  __shared__ double next_c;
  __shared__ unsigned flags;
  __shared__ float wmax[32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  // ---- pairwise sum: the levels above replay_sum_leaves' CTAs
  const int P = 1 << top_levels;
  for (int k = tid; k < P; k += kDrawThreads) {
    tv[k] = part[k];
    te[k] = part_exists[k];
  }
  if (tid == 0) flags = 0u;
  __syncthreads();
  for (int w = P / 2; w >= 1; w >>= 1) {
    float r[(1 << kTopBits) / 2 / kDrawThreads + 1];
    uint8_t e[(1 << kTopBits) / 2 / kDrawThreads + 1];
    int c = 0;
    for (int k = tid; k < w; k += kDrawThreads, ++c) {
      e[c] = te[2 * k];
      r[c] = te[2 * k + 1] ? __fadd_rn(tv[2 * k], tv[2 * k + 1]) : tv[2 * k];
    }
    __syncthreads();
    c = 0;
    for (int k = tid; k < w; k += kDrawThreads, ++c) {
      tv[k] = r[c];
      te[k] = e[c];
    }
    __syncthreads();
  }
  const float s = tv[0];

  // ---- exact cumulative sum of p = float64(q / s), stretch by stretch
  unsigned my_flags = 0u;  // HMZ_REPLAY_NAN: a NaN row; HMZ_REPLAY_NEGATIVE: p < 0; bit 8: an infinite row before the last
  double c = 0.0;
  for (int64_t pos = 0; pos < num;) {
    double xs[kItems];
#pragma unroll
    for (int j = 0; j < kItems; ++j) {
      const int64_t g = pos + (int64_t)tid * kItems + j;
      double x = 0.0;
      if (g < num) {
        const float xf = __fdiv_rn(q[g], s);
        if (xf != xf) my_flags |= HMZ_REPLAY_NAN;
        if (xf < 0.0f) my_flags |= HMZ_REPLAY_NEGATIVE;
        if (isinf(xf) && g < num - 1) my_flags |= 256u;
        if (xf > 0.0f && !isinf(xf)) x = (double)xf;  // what the scan adds; rows it skips only occur in rings NumPy rejects
      }
      xs[j] = x;
    }
    int first = INT_MAX;
    if (c == 0.0) {  // leading zero rows: c stays 0 up to the first non-zero row, which sets it exactly
#pragma unroll
      for (int j = 0; j < kItems; ++j)
        if (xs[j] > 0.0 && first == INT_MAX) first = tid * kItems + j;
      const int k = block_min(first, red);
#pragma unroll
      for (int j = 0; j < kItems; ++j) {
        const int local = tid * kItems + j;
        const int64_t g = pos + local;
        if (g < num && local <= k) cdf[g] = local == k ? xs[j] : 0.0;
        if (local == k) next_c = xs[j];
      }
      __syncthreads();
      if (k != INT_MAX) c = next_c;
      pos += k == INT_MAX ? kChunk : (int64_t)k + 1;
      __syncthreads();
      continue;
    }
    const unsigned long long cb = (unsigned long long)__double_as_longlong(c);
    const int E = (int)(cb >> 52);
    const unsigned long long C0 = (cb & ((1ull << 52) - 1)) | (1ull << 52);
    const unsigned b0 = (unsigned)(C0 & 1ull);
    // c / u entering this thread's first row: a scan of the row maps over the chunk.  Chunks without a tie (the common
    // case) scan plain increments; otherwise the parity-dependent maps are composed.
    bool tie = false;
    unsigned long long plain = 0;
#pragma unroll
    for (int j = 0; j < kItems; ++j) {
      unsigned long long n;
      int cls;
      row_parts(xs[j], E, n, cls);
      tie |= cls == 2;
      plain = sat_add(plain, sat_add(n, (unsigned long long)(cls & 1)));
    }
    unsigned long long pre_inc;
    if (__syncthreads_or(tie)) {
      RowMap agg = identity_map();
#pragma unroll
      for (int j = 0; j < kItems; ++j) agg = compose(agg, row_map(xs[j], E));
      RowMap inc = agg;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const RowMap o = shfl_up_map(inc, d);
        if (lane >= d) inc = compose(o, inc);
      }
      if (lane == 31) warp_maps[warp] = inc;
      RowMap pre = shfl_up_map(inc, 1);
      if (lane == 0) pre = identity_map();
      __syncthreads();
      if (warp == 0) {
        RowMap wm = warp_maps[lane];
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
          const RowMap o = shfl_up_map(wm, d);
          if (lane >= d) wm = compose(o, wm);
        }
        warp_maps[lane] = wm;  // inclusive over warps
      }
      __syncthreads();
      if (warp > 0) pre = compose(warp_maps[warp - 1], pre);
      pre_inc = b0 ? pre.inc1 : pre.inc0;
    } else {
      unsigned long long inc = plain;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const unsigned long long o = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc = sat_add(o, inc);
      }
      if (lane == 31) warp_incs[warp] = inc;
      unsigned long long pre = __shfl_up_sync(0xffffffffu, inc, 1);
      if (lane == 0) pre = 0;
      __syncthreads();
      if (warp == 0) {
        unsigned long long wi = warp_incs[lane];
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
          const unsigned long long o = __shfl_up_sync(0xffffffffu, wi, d);
          if (lane >= d) wi = sat_add(o, wi);
        }
        warp_incs[lane] = wi;
      }
      __syncthreads();
      pre_inc = warp > 0 ? sat_add(warp_incs[warp - 1], pre) : pre;
    }
    // first row whose sum reaches the next binade (c / u >= 2^53)
    unsigned long long v = C0 + pre_inc;
#pragma unroll
    for (int j = 0; j < kItems; ++j) {
      if (v >= kTop) break;
      unsigned long long n;
      int cls;
      row_parts(xs[j], E, n, cls);
      v = row_add(v, n, cls);
      if (v >= kTop) first = tid * kItems + j;
    }
    const int k = block_min(first, red);
    v = C0 + pre_inc;
    const int last_local = (int)((num - pos < kChunk ? num - pos : kChunk) - 1);
#pragma unroll
    for (int j = 0; j < kItems; ++j) {
      const int local = tid * kItems + j;
      const int64_t g = pos + local;
      if (g >= num || local > k) break;
      unsigned long long n;
      int cls;
      row_parts(xs[j], E, n, cls);
      const unsigned long long val = row_add(v, n, cls);
      double cv;
      if (local < k) {
        cv = make_c(E, val);
      } else {  // the row that leaves the binade: exact when it lands on 2^(e+1), else one ordinary add
        cv = val == kTop ? make_c(E, val) : __dadd_rn(make_c(E, v), xs[j]);
        next_c = cv;
      }
      cdf[g] = cv;
      if (k == INT_MAX && local == last_local) next_c = cv;
      v = val;
    }
    __syncthreads();
    c = next_c;
    pos += k == INT_MAX ? kChunk : (int64_t)k + 1;
    __syncthreads();
  }

  // ---- NumPy's checks, in its order of evaluation (the status word only accumulates bits)
  my_flags = __reduce_or_sync(0xffffffffu, my_flags);
  if (lane == 0 && my_flags) atomicOr(&flags, my_flags);
  __syncthreads();
  const double c_last = cdf[num - 1];
  if (tid == 0) {
    unsigned f = flags & (HMZ_REPLAY_NAN | HMZ_REPLAY_NEGATIVE);
    bool any_inf = (flags & 256u) != 0;
    double ksum = 0.0;
    if (num <= 2) {  // kahan_sum(p) literally: its NaN / inf outcome with infinite rows depends on their position
      ksum = (double)__fdiv_rn(q[0], s);
      double cc = 0.0;
      for (int64_t i = 1; i < num; ++i) {
        const double y = __dsub_rn((double)__fdiv_rn(q[i], s), cc);
        const double t = __dadd_rn(ksum, y);
        cc = __dsub_rn(__dsub_rn(t, ksum), y);
        ksum = t;
      }
      f = (f & ~HMZ_REPLAY_NAN) | (ksum != ksum ? HMZ_REPLAY_NAN : 0u);
    } else {
      // an infinite row before the last turns Kahan's compensation into NaN; one in the last row gives an infinite sum
      if (any_inf) f |= HMZ_REPLAY_NAN;
      const double last = (double)__fdiv_rn(q[num - 1], s);
      ksum = isinf(last) ? last : c_last;
    }
    // The sum check uses the cumulative sum's last value (what cdf /= cdf[-1] divides by) instead of Kahan's sum: they
    // differ by at most num * 2^-53, so only a sum within ~1e-10 (at a million rows) of the threshold could be judged
    // differently.  Float32 rounding of q / s moves the sum by ~1e-6.
    if (!(f & HMZ_REPLAY_NAN) && fabs(ksum - 1.0) > kSumAtol) f |= HMZ_REPLAY_SUM;
    if (f) atomicOr(status, (int32_t)f);
  }

  // ---- searchsorted(cdf / cdf[-1], u, side="right") and the importance weights
  float my_max = -INFINITY;
  for (int64_t j = tid; j < batch; j += kDrawThreads) {
    const double u = uniforms[j];
    int64_t lo = 0, hi = num;
    while (lo < hi) {
      const int64_t mid = (lo + hi) >> 1;
      if (__ddiv_rn(cdf[mid], c_last) > u)
        hi = mid;
      else
        lo = mid + 1;
    }
    if (lo > num - 1) lo = num - 1;  // only in rings NumPy rejects (NaN cdf)
    indices[j] = lo;
    float w = __fdiv_rn(inv_size, __fdiv_rn(q[lo], s));
    if (beta == 0.0f)
      w = 1.0f;  // NumPy's power: x ** 0 = ones_like(x)
    else if (beta == 0.5f)
      w = __fsqrt_rn(w);  // x ** 0.5 = sqrt(x)
    else if (beta == 2.0f)
      w = __fmul_rn(w, w);
    else if (beta == -1.0f)
      w = __fdiv_rn(1.0f, w);
    else if (beta != 1.0f)
      w = powf(w, beta);
    weights[j] = w;
    my_max = nan_max(my_max, w);
  }
  for (int d = 16; d >= 1; d >>= 1) my_max = nan_max(my_max, __shfl_xor_sync(0xffffffffu, my_max, d));
  if (lane == 0) wmax[warp] = my_max;
  __syncthreads();
  float mx = wmax[0];
  for (int k = 1; k < kDrawThreads / 32; ++k) mx = nan_max(mx, wmax[k]);
  for (int64_t j = tid; j < batch; j += kDrawThreads) weights[j] = __fdiv_rn(weights[j], mx);
}

// update_priorities: assert all finite and at least one > 0, then priorities[indices] = new_priorities with the last
// occurrence of a repeated index winning, as NumPy's fancy assignment does.
__global__ void __launch_bounds__(1024) replay_set_priorities(float* __restrict__ priorities, int64_t size,
                                                             const int64_t* __restrict__ indices, const float* __restrict__ new_p,
                                                             int64_t batch, int32_t* __restrict__ status) {
  int bad = 0, positive = 0;
  for (int64_t j = threadIdx.x; j < batch; j += blockDim.x) {
    const float v = new_p[j];
    bad |= !isfinite(v);
    positive |= v > 0.0f;
  }
  bad = __syncthreads_or(bad);
  positive = __syncthreads_or(positive);
  if (bad || !positive) {
    if (threadIdx.x == 0) atomicOr(status, (int32_t)HMZ_REPLAY_PRIORITY);
    return;
  }
  for (int64_t j = threadIdx.x; j < batch; j += blockDim.x) {
    const int64_t i = indices[j];
    if (i < 0 || i >= size) continue;
    bool last = true;
    for (int64_t k = j + 1; k < batch && last; ++k) last = indices[k] != i;
    if (last) priorities[i] = new_p[j];
  }
}

struct Workspace {
  double* cdf;
  float* part;
  uint8_t* part_exists;
  int depth;
};

int64_t align256(int64_t b) { return (b + 255) & ~(int64_t)255; }

Workspace workspace_layout(void* base, int64_t num) {
  Workspace w;
  w.depth = pairwise_depth(num);
  if (w.depth < 8) w.depth = 8;
  const int64_t parts = (int64_t)1 << (w.depth - 8);
  char* p = (char*)base;
  w.cdf = (double*)p;
  p += align256(num * (int64_t)sizeof(double));
  w.part = (float*)p;
  p += align256(parts * (int64_t)sizeof(float));
  w.part_exists = (uint8_t*)p;
  return w;
}

constexpr int64_t kMaxRows = (int64_t)1 << 27;

}  // namespace
}  // namespace hmz

using namespace hmz;

extern "C" {

int64_t hmz_replay_sample_workspace_bytes(int64_t num) {
  if (num < 1 || num > kMaxRows) return 0;
  int d = pairwise_depth(num);
  if (d < 8) d = 8;
  const int64_t parts = (int64_t)1 << (d - 8);
  return align256(num * (int64_t)sizeof(double)) + align256(parts * (int64_t)sizeof(float)) + align256(parts);
}

int hmz_replay_sample(const float* priorities, int64_t num, int64_t size, double priority_exponent, const double* uniforms,
                      int64_t batch, double importance_exponent, void* workspace, int64_t* indices, float* weights, int32_t* status,
                      void* stream) {
  ProfScope prof_scope(HMZ_PROF_OTHER, stream);
  if (!priorities || !uniforms || !workspace || !indices || !weights || !status)
    return fail(HMZ_ERR_INVALID, "hmz_replay_sample: null pointer");
  if (num < 1 || size < num || batch < 1)
    return fail(HMZ_ERR_INVALID, "hmz_replay_sample: need 1 <= num <= size and batch >= 1 (num=%lld size=%lld batch=%lld)",
                (long long)num, (long long)size, (long long)batch);
  if (!isfinite(importance_exponent)) return fail(HMZ_ERR_INVALID, "hmz_replay_sample: importance exponent is not finite");
  if (priority_exponent != 1.0)
    return fail(HMZ_ERR_UNSUPPORTED, "hmz_replay_sample: priority exponent %g (only 1 is sampled on the device)", priority_exponent);
  if (num > kMaxRows) return fail(HMZ_ERR_UNSUPPORTED, "hmz_replay_sample: %lld rows (at most 2^27)", (long long)num);
  const Workspace w = workspace_layout(workspace, num);
  if (w.depth - 8 > kTopBits) return fail(HMZ_ERR_UNSUPPORTED, "hmz_replay_sample: pairwise tree too deep");
  const cudaStream_t s = (cudaStream_t)stream;
  replay_sum_leaves<<<(unsigned)(1u << (w.depth - 8)), kSumThreads, 0, s>>>(priorities, num, w.depth, w.part, w.part_exists);
  int rc = check_launch("replay_sum_leaves");
  if (rc != HMZ_OK) return rc;
  // (1.0 / self.size) is a Python float; NumPy 2 casts it to float32 against the float32 probabilities
  const float inv_size = (float)(1.0 / (double)size);
  replay_draw<<<1, kDrawThreads, 0, s>>>(priorities, num, w.depth - 8, w.part, w.part_exists, w.cdf, uniforms, batch, inv_size,
                                         (float)importance_exponent, indices, weights, status);
  return check_launch("replay_draw");
}

int hmz_replay_set_priorities(float* priorities, int64_t size, const int64_t* indices, const float* new_priorities, int64_t batch,
                              int32_t* status, void* stream) {
  ProfScope prof_scope(HMZ_PROF_OTHER, stream);
  if (!priorities || !indices || !new_priorities || !status) return fail(HMZ_ERR_INVALID, "hmz_replay_set_priorities: null pointer");
  if (size < 1 || batch < 1) return fail(HMZ_ERR_INVALID, "hmz_replay_set_priorities: need size >= 1 and batch >= 1");
  replay_set_priorities<<<1, 1024, 0, (cudaStream_t)stream>>>(priorities, size, indices, new_priorities, batch, status);
  return check_launch("replay_set_priorities");
}

}  // extern "C"
