// MuZeroNet inference on the 5th-generation tensor cores (HMZ_MODE_BF16): recurrent_inference
// (networks.py:96-116: dynamics :129-138, prediction :140-150) and initial_inference (:71-94:
// represent :124-127, prediction), both with the support transform (:152-189) and normalize_h_state
// (:191-196), as ONE persistent kernel template.
//
// One CTA pass = two tiles of 128 rows (UMMA M = 128, cta_group::1), ping-ponged; per tile and network
//   first layer   H[0:256) = [A | AX] x [W1 | W1_action, b1]^T    tcgen05.mma kind::f16 (bf16 x bf16 -> fp32 in TMEM)
//                 A  = input latent / one-hot observation / new latent tile in shared memory (K-major, SWIZZLE_128B)
//                 AX = [onehot(action) (6), 1, 0 x 9] per row (K = 16): every bias and the one-hot action columns
//                      of dynamic_net.0 ride in this extra MMA step, so no epilogue does bias arithmetic
//   epilogue      tcgen05.ld -> relu + bf16 (one cvt.rn.relu.bf16x2 per pair) -> tcgen05.st IN PLACE: the hidden
//                 activations never leave TMEM
//   second layer  O = [A1 | AX] x [W2 | b2]^T with A1 taken from TMEM (the .ts form of tcgen05.mma)
//   latent        min-max normalised in registers -> raw / normalised bf16 tiles (the heads' A operands) + HBM
//   heads         softmax expectation over the 33-bin support + signed parabolic, policy softmax, in registers
//
// Weights (pre-swizzled by hmz_weights_pack into the exact shared-memory image, with the extra slice
// appended) are streamed from L2 per layer with 1-D TMA bulk copies (cp.async.bulk + mbarrier
// complete_tx) by a loader warp into double-buffered slots that BOTH tiles consume.
#include <cstdlib>
#include <cstring>
#include <vector>

#include "hmz_net_tc.cuh"

namespace hmz {

namespace tc {
namespace v4 {
// The stand-alone kernels: one launch per network evaluation of a whole batch (grid = min(tile pairs, SMs)).
template <bool kInitial>
__global__ void __launch_bounds__(kLaunchThreads, 1) net_tc(const __grid_constant__ TcArgs a) {
  extern __shared__ uint8_t smem_raw[];
  net_tc_body<kInitial, false>(a, PersistCtl{}, smem_raw, (int)blockIdx.x, (int)gridDim.x);
}
}  // namespace v4

// ---- host-side packing ----------------------------------------------------------------
static uint16_t f2bf(float f) {
  uint32_t u;
  std::memcpy(&u, &f, 4);
  if ((u & 0x7FFFFFFFu) > 0x7F800000u) return (uint16_t)((u >> 16) | 0x40u);  // NaN
  return (uint16_t)((u + 0x7FFFu + ((u >> 16) & 1u)) >> 16);
}

// torch Linear weight w [out][in] (row-major) restricted to input columns [k0, k0 + 64*k_atoms) ->
// k_atoms SWIZZLE_128B K-atoms of [out_pad rows][128 B]; rows >= out are zero.
static void pack_kmajor_sw128(uint8_t* dst, const float* w, int out, int in, int out_pad, int k0, int k_atoms) {
  for (int ka = 0; ka < k_atoms; ++ka)
    for (int n = 0; n < out_pad; ++n)
      for (int c = 0; c < 8; ++c) {
        uint16_t* chunk = reinterpret_cast<uint16_t*>(dst + (size_t)ka * out_pad * 128 + (size_t)n * 128 + ((c ^ (n & 7)) << 4));
        for (int j = 0; j < 8; ++j) {
          const int k = k0 + ka * 64 + c * 8 + j;
          chunk[j] = (n < out && k < in) ? f2bf(w[(size_t)n * in + k]) : (uint16_t)0;
        }
      }
}
}  // namespace tc

// bf16 blob = [tensor-core section, fixed size][float32 blob of hmz_net.cu]: the section comes first
// so that the recurrent path needs no disk count to find it.
int64_t tc_fp32_offset_bytes() { return ((int64_t)tc::kSectionBytes + 1023) / 1024 * 1024; }

int64_t tc_packed_bytes(int n_disks) { return tc_fp32_offset_bytes() + (int64_t)Fp32Layout::total(n_disks) * 4; }

// extra K = 16 slice of a weight block in the core-matrix layout: column kBiasK carries the bias,
// columns 0..n_extra-1 carry w[:, extra_col0 + j] (the one-hot action columns of dynamic_net.0).
static void pack_extra(uint8_t* dst, const float* w, const float* bias, int out, int in, int out_pad, int extra_col0,
                       int n_extra) {
  for (int n = 0; n < out_pad; ++n)
    for (int c = 0; c < 2; ++c) {
      uint16_t* chunk = reinterpret_cast<uint16_t*>(dst + tc::plain_off(n, c));
      for (int j = 0; j < 8; ++j) {
        const int k = c * 8 + j;
        float v = 0.f;
        if (n < out) {
          if (k < n_extra) v = w[(size_t)n * in + extra_col0 + k];
          else if (k == tc::kBiasK) v = bias[n];
        }
        chunk[j] = tc::f2bf(v);
      }
    }
}

void tc_pack(const float* const* t, int n_disks, void* out) {
  using namespace tc;
  std::memset(out, 0, (size_t)tc_packed_bytes(n_disks));
  // the root inference (1/S of the work) runs on the float32 copy behind the section
  pack_fp32(t, n_disks, (float*)((uint8_t*)out + tc_fp32_offset_bytes()));
  uint8_t* sec = (uint8_t*)out;
  // state_dict order: rep(0-3) dyn(4-7) rwd(8-11) pol(12-15) val(16-19); each {w1, b1, w2, b2}
  const int in_g1 = kLatent + kActions;
  pack_kmajor_sw128(sec + kWg1, t[4], kHidden, in_g1, 256, 0, 1);
  pack_extra(sec + kWg1 + 256 * 128, t[4], t[5], kHidden, in_g1, 256, kLatent, kActions);
  pack_kmajor_sw128(sec + kWg2, t[6], kLatent, kHidden, 64, 0, 4);
  pack_extra(sec + kWg2 + 64 * 128 * 4, t[6], t[7], kLatent, kHidden, 64, 0, 0);
  // representation_net (root inference): Linear(3N, 256) on the one-hot observation padded to K = 64, Linear(256, 64)
  pack_kmajor_sw128(sec + kWh1, t[0], kHidden, 3 * n_disks, 256, 0, 1);
  pack_extra(sec + kWh1 + 256 * 128, t[0], t[1], kHidden, 3 * n_disks, 256, 0, 0);
  pack_kmajor_sw128(sec + kWh2, t[2], kLatent, kHidden, 64, 0, 4);
  pack_extra(sec + kWh2 + 64 * 128 * 4, t[2], t[3], kLatent, kHidden, 64, 0, 0);
  const struct { uint32_t w1, w2; int i; int out2, pad2; } heads[3] = {
      {kWr1, kWr2, 8, kSupport, 48}, {kWp1, kWp2, 12, kActions, 16}, {kWv1, kWv2, 16, kSupport, 48}};
  for (const auto& h : heads) {
    pack_kmajor_sw128(sec + h.w1, t[h.i], kHidden, kLatent, 256, 0, 1);
    pack_extra(sec + h.w1 + 256 * 128, t[h.i], t[h.i + 1], kHidden, kLatent, 256, 0, 0);
    pack_kmajor_sw128(sec + h.w2, t[h.i + 2], h.out2, kHidden, h.pad2, 0, 4);
    pack_extra(sec + h.w2 + h.pad2 * 128 * 4, t[h.i + 2], t[h.i + 3], h.out2, kHidden, h.pad2, 0, 0);
  }
}

static int tc_timeline_enabled() {
  static const int on = getenv("HMZ_TC_TIMELINE") ? atoi(getenv("HMZ_TC_TIMELINE")) : 0;
  return on;
}

int tc_debug_read_timeline(unsigned long long* host_out) {
  return cudaMemcpyFromSymbol(host_out, tc::g_timeline, sizeof(unsigned long long) * 96) == cudaSuccess ? HMZ_OK : HMZ_ERR_CUDA;
}

static int tc_prepare(int* smem_bytes) {
  static thread_local int done_dev = -1;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return fail(HMZ_ERR_CUDA, "cudaGetDevice failed (no CUDA device?)");
  *smem_bytes = (int)sizeof(tc::v4::Smem) + 1024;
  if (done_dev != dev) {
    cudaError_t e = cudaFuncSetAttribute(tc::v4::net_tc<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, *smem_bytes);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(tc::v4::net_tc<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, *smem_bytes);
    if (e != cudaSuccess) return fail(HMZ_ERR_CUDA, "cudaFuncSetAttribute(net_tc): %s", cudaGetErrorString(e));
    done_dev = dev;
  }
  return HMZ_OK;
}

// One tile pair per CTA while there are SMs for it (DESIGN §9: two passes per CTA did not pay).
static unsigned tc_grid(int64_t n, int* n_pairs) {
  const int64_t pairs = (n + 2 * tc::kM - 1) / (2 * tc::kM);
  const int sms = sm_count();
  *n_pairs = (int)pairs;
  return (unsigned)(pairs < sms ? pairs : sms);
}

int tc_net_recurrent(const void* weights, const void* lat_in, int64_t in_rows_per_item, const uint16_t* in_row,
                     const uint8_t* actions, void* lat_out, int64_t out_rows_per_item, int64_t out_row,
                     int latent_dtype, float* r, float* p, float* v, int64_t n, cudaStream_t stream, const uint16_t* block_set,
                     int64_t weight_stride, bool allow_head_split) {
  int smem = 0, n_pairs = 0;
  if (int rc = tc_prepare(&smem)) return rc;
  unsigned grid = tc_grid(n, &n_pairs);
  tc::v4::TcArgs a{};
  // small batches: three CTAs per tile pair, one head each (TcArgs::head_split)
  a.head_split = (allow_head_split && 3 * n_pairs <= sm_count()) ? 3 : 1;
  if (a.head_split == 3) grid = 3u * (unsigned)n_pairs;
  a.wsec = (const uint8_t*)weights;
  a.block_set = block_set;
  a.weight_stride = weight_stride;
  a.lat_in = lat_in;
  a.in_rows_per_item = in_rows_per_item;
  a.in_row = in_row;
  a.actions = actions;
  a.lat_out = lat_out;
  a.out_rows_per_item = out_rows_per_item;
  a.out_row = out_row;
  a.latent_dtype = latent_dtype;
  a.r_out = r;
  a.p_out = p;
  a.v_out = v;
  a.n = n;
  a.n_pairs = n_pairs;
  a.timeline = tc_timeline_enabled();
  a.gantt = gantt_next(0, gantt_context_tag());
  cudaError_t e = launch_pdl(tc::v4::net_tc<false>, dim3(grid), dim3(tc::v4::kLaunchThreads), (size_t)smem, stream, a);
  if (e != cudaSuccess) return fail(HMZ_ERR_CUDA, "net_tc<recurrent> launch: %s", cudaGetErrorString(e));
  return check_launch("net_tc<recurrent>");
}

int tc_net_initial(const void* weights, int n_disks, const uint32_t* words, void* lat_out, int64_t out_rows_per_item,
                   int latent_dtype, float* p0, float* v0, int64_t n, cudaStream_t stream, const uint16_t* block_set,
                   int64_t weight_stride) {
  int smem = 0, n_pairs = 0;
  if (int rc = tc_prepare(&smem)) return rc;
  const unsigned grid = tc_grid(n, &n_pairs);
  tc::v4::TcArgs a{};
  a.wsec = (const uint8_t*)weights;
  a.block_set = block_set;
  a.weight_stride = weight_stride;
  a.in_rows_per_item = 1;
  a.words = words;
  a.n_disks = n_disks;
  a.lat_out = lat_out;
  a.out_rows_per_item = out_rows_per_item;
  a.out_row = 0;
  a.latent_dtype = latent_dtype;
  a.p_out = p0;
  a.v_out = v0;
  a.n = n;
  a.n_pairs = n_pairs;
  a.head_split = 1;
  cudaError_t e = launch_pdl(tc::v4::net_tc<true>, dim3(grid), dim3(tc::v4::kLaunchThreads), (size_t)smem, stream, a);
  if (e != cudaSuccess) return fail(HMZ_ERR_CUDA, "net_tc<initial> launch: %s", cudaGetErrorString(e));
  return check_launch("net_tc<initial>");
}

}  // namespace hmz
