// MuZeroNet recurrent_inference (networks.py:96-116) and initial_inference (:71-94) at float32 accuracy ON THE TENSOR
// CORES (HMZ_MODE_FP32X3): the fast parity mode.  Every float32 operand is split into three bf16 parts, x = x0 + x1 + x2 with
// x0 = bf16(x), x1 = bf16(x - x0), x2 = bf16(x - x0 - x1) (the residuals are exact in float32), and a product
// x w is evaluated as the seven bf16 x bf16 products x0 w0, x1 w0, x2 w0, x0 w1, x1 w1, x2 w1, x0 w2 — each
// exact in the float32 accumulator; the dropped x1 w2, x2 w2 are <= 2^-25 |x w|.  Per Linear layer that is
//     D[:, 0:n)  = (x0 + x1 + x2) w0^T          tcgen05.mma kind::f16, one N = 2n instruction per part and k-step
//     D[:, n:2n) = (x0 + x1 + x2) w1^T + x0 w2^T    (+ one N = n instruction per k-step for the w2 term)
// with the weight parts stacked along N in shared memory ([w0; w1; w2] rows of one SWIZZLE_128B K-atom), and the
// epilogue adds the two accumulator blocks.  The small terms accumulate apart from the large one, so the
// accumulator's rounding acts on them at their own scale.
//
// One CTA = one tile of 128 rows (UMMA M = 128), persistent over tiles.  A network is processed in four CHUNKS
// of 64 hidden units: first layer of chunk c -> TMEM accumulator (128 columns, two buffers) -> the hidden-epilogue
// warps add the blocks, apply relu, split into three bf16 parts and write them back IN PLACE -> the second layer
// accumulates the chunk's K = 64 slice with its A operand taken from TMEM (the .ts form).  Separate issuing warps for
// the layer kinds (two alternating on the first layers, one for the second: issuing a tcgen05.mma blocks for about its
// execution time), so first layers run ahead of second layers and the tensor core works while a chunk is drained; four
// output warps (thread = row) own the new latent, the heads' outputs and the gather of the next tile.  Bias and the one-hot action columns of dynamic_net.0 ride in an extra K = 16 step
// as in the bf16 kernel (hmz_net_tc.cuh).  Weights stream from L2 per chunk with 1-D TMA bulk copies into
// double-buffered slots.  Small batches (3 x tiles <= SMs): three CTAs per tile run
// the dynamics network and ONE head each.  Epilogue math (normalize_h_state :191-196, support transform :152-189,
// softmax) is the float32 code of the FFMA kernel (hmz_net.cu).  DESIGN.md §4 has the measurements.
#include <cstdlib>
#include <cstring>

#include "hmz_net_tc.cuh"

namespace hmz {
namespace x3 {
using namespace tc;
using tc::v4::tmem_ld16_issue;
using tc::v4::tmem_ld16_wait;
using tc::v4::tmem_st8;
using tc::v4::tmem_st_wait;
using tc::v4::umma_ts;

constexpr int kEpiThreads = 256;  // 8 hidden-epilogue warps: warp -> TMEM lane quarter (w & 3), column half (w >> 2)
constexpr int kOutThreads = 128;  // 4 output warps: thread = row
constexpr int kOutWarp0 = 8, kMma1Warp = 12, kMma1bWarp = 13, kMma2Warp = 14, kLoaderWarp = 15;
constexpr int kThreads = 16 * 32;
constexpr uint32_t kW1Main = 192 * 128;            // [w0; w1; w2] rows of a 64-unit chunk, K = 64
constexpr uint32_t kW1Bytes = 192 * 160;           // + the extra K = 16 slice
constexpr uint32_t kSlot = 30720;                  // both layer kinds: 192 x 160 >= 3 n2 x 160
constexpr uint32_t kBlockStride = 2 * kSlot;       // one (network, chunk) block of the weight section
constexpr uint32_t kRepBlock0 = 16;                // blocks 16..19: representation_net (root inference)
constexpr uint32_t kSectionBytes = 20 * kBlockStride;
constexpr uint32_t kBufs = 2;                      // first-layer accumulator buffers
constexpr uint32_t kColD2 = 128 * kBufs;           // TMEM: D1[2] at columns 0 / 128, D2 at 256,
constexpr uint32_t kColHn = kColD2 + 128;          //       the normalised latent's three bf16 parts at 384 + 32 part (96 columns)
// second-layer width per network in pass order dynamics, reward, value, policy (33 support logits -> 48, 6 -> 16)
__host__ __device__ constexpr uint32_t n2_of(int net) { return net == 0 ? 64u : (net == 3 ? 16u : 48u); }

struct __align__(1024) Smem {
  uint8_t t0[3][kAtomA];  // parts of the input latent tile, later of the raw new latent (reward head input)
  uint8_t w1[2][kSlot];   // first-layer chunk blocks, slot = chunk counter & 1
  uint8_t w2[2][kSlot];   // second-layer chunk blocks
  uint8_t ax[kM * 32];    // extra A slice [onehot(action) (6), 1, 0 x 9] per row (exact in bf16: one part)
  uint64_t bar_w1full[2], bar_w1free[2], bar_w2full[2], bar_w2free[2];
  uint64_t bar_g;         // input tile + extra slice written (128 arrivals: the output warps)
  uint64_t bar_g0;        // the same for the CTA's FIRST tile, which the idle hidden-epilogue warps gather (256 + 128 arrivals)
  uint64_t bar_d[kBufs];      // first-layer accumulator of the buffer complete
  uint64_t bar_a[kBufs];      // hidden parts written back (256 arrivals)
  uint64_t bar_hfree[kBufs];  // the second layer that read the buffer's hidden parts has completed
  uint64_t bar_o;         // second layer of a network complete
  uint64_t bar_raw;       // dynamics output: D2 drained and the raw latent tile written (128 arrivals)
  uint64_t bar_hn;        // dynamics output: normalised latent parts written to TMEM (128 arrivals)
  uint64_t bar_out;       // a head's output: D2 drained (128 arrivals)
  uint32_t tmem_base;
};

struct Args {
  const uint8_t* wsec;
  const void* lat_in;
  int64_t in_rows_per_item;
  const uint16_t* in_row;
  const uint8_t* actions;
  const uint32_t* words;  // env words (initial inference)
  int n_disks;
  void* lat_out;
  int64_t out_rows_per_item, out_row;
  int latent_dtype;
  float *r_out, *p_out, *v_out;
  int64_t n;
  int n_tiles;
  int head_split;  // 3: small batches (3 x tiles <= SMs) — CTAs 3 t, 3 t + 1, 3 t + 2 all run the dynamics network of tile t and
                   // then ONE head each (reward + the latent rows / value / policy), as in the bf16 kernel: the dependent chain
                   // of a launch shrinks from sixteen chunks to eight while idle SMs do the redundant work; else 1
  int timeline;  // tooling (HMZ_X3_TIMELINE=1): CTA 0 records clock64() at the phase boundaries of its first tile
  const uint16_t* block_set;  // nullable: weight set of each 256-row block (hmz_multi_t), at wsec + block_set[tile / 2] * weight_stride
  int64_t weight_stride;
};

static __device__ unsigned long long g_x3_timeline[160];
#define X3_TL(slot)                                                   \
  do {                                                                \
    if (tl_on) {                                                      \
      unsigned long long now_;                                        \
      asm volatile("mov.u64 %0, %%clock64;" : "=l"(now_)::"memory");  \
      g_x3_timeline[slot] = now_;                                     \
    }                                                                 \
  } while (0)

// Every wait of this kernel is time-bounded (2 s: a launch lasts well under a millisecond): a protocol failure traps —
// the launch fails with an error — instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
  uint32_t spins = 0;
  unsigned long long t0 = 0;
  for (;;) {
    uint32_t ok;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}"
        : "=r"(ok)
        : "r"(addr), "r"(parity)
        : "memory");
    if (ok) return;
    if ((++spins & 0xFFFu) == 0u) {
      const unsigned long long now = globaltimer_ns();
      if (t0 == 0) t0 = now;
      else if (now - t0 > 2000000000ull) __trap();
    }
  }
}

__device__ __forceinline__ float bf_lo(uint32_t p) { return __uint_as_float(p << 16); }
__device__ __forceinline__ float bf_hi(uint32_t p) { return __uint_as_float(p & 0xFFFF0000u); }
// three bf16 parts of two floats (a in the low half-words)
__device__ __forceinline__ void split3(float a, float b, uint32_t& p0, uint32_t& p1, uint32_t& p2) {
  p0 = pack_bf16(a, b);
  a = __fsub_rn(a, bf_lo(p0));
  b = __fsub_rn(b, bf_hi(p0));
  p1 = pack_bf16(a, b);
  a = __fsub_rn(a, bf_lo(p1));
  b = __fsub_rn(b, bf_hi(p1));
  p2 = pack_bf16(a, b);
}
// eight floats -> the 16-byte chunk `chunk` of row `row` in the three part tiles
__device__ __forceinline__ void store_parts8(uint8_t (*tile)[kAtomA], int row, int chunk, const float (&x)[8]) {
  uint32_t p[3][4];
#pragma unroll
  for (int j = 0; j < 4; ++j) split3(x[2 * j], x[2 * j + 1], p[0][j], p[1][j], p[2][j]);
  const uint32_t addr = smem_u32(tile[0]) + sw128(row, chunk);  // (explicit st.shared: the pointer form compiles to generic stores)
#pragma unroll
  for (int i = 0; i < 3; ++i)
    asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(addr + (uint32_t)i * kAtomA), "r"(p[i][0]), "r"(p[i][1]), "r"(p[i][2]),
                 "r"(p[i][3])
                 : "memory");
}
// out[j] = block 0 column j + block 1 column j for 16 columns (the two accumulator blocks of a layer)
__device__ __forceinline__ void ld_sum16(uint32_t t0, uint32_t t1, float (&out)[16]) {
  uint32_t a[16], b[16];
  tmem_ld16_issue(t0, a);
  tmem_ld16_issue(t1, b);
  tmem_ld16_wait(a);
  tmem_ld16_wait(b);
#pragma unroll
  for (int j = 0; j < 16; ++j) out[j] = __fadd_rn(__uint_as_float(a[j]), __uint_as_float(b[j]));
}

__device__ __forceinline__ void tmem_st4(uint32_t taddr, const uint32_t (&r)[4]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};" ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]) : "memory");
}

// Hidden epilogue of one chunk for this thread's row and column half: units 32 half .. 32 half + 31 of the chunk.
// Batch b (16 units) reads columns [16b, 16b + 16) of both blocks and leaves h0 in [16b, 16b + 8), h1 in
// [16b + 8, 16b + 16) and h2 in [64 + 16b, 64 + 16b + 8): always inside the columns it has just read.
__device__ __forceinline__ void hidden_epilogue(uint32_t D, int half) {
  uint32_t a[2][16], b[2][16];
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    tmem_ld16_issue(D + 32 * half + 16 * j, a[j]);
    tmem_ld16_issue(D + 64 + 32 * half + 16 * j, b[j]);
  }
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    tmem_ld16_wait(a[j]);
    tmem_ld16_wait(b[j]);
  }
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    uint32_t p0[8], p1[8], p2[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const float lo = fmaxf(__fadd_rn(__uint_as_float(a[j][2 * i]), __uint_as_float(b[j][2 * i])), 0.f);
      const float hi = fmaxf(__fadd_rn(__uint_as_float(a[j][2 * i + 1]), __uint_as_float(b[j][2 * i + 1])), 0.f);
      split3(lo, hi, p0[i], p1[i], p2[i]);
    }
    const uint32_t c = D + 32 * half + 16 * j;
    tmem_st8(c, p0);
    tmem_st8(c + 8, p1);
    tmem_st8(c + 64, p2);
  }
  tmem_st_wait();
}

// Parent latents (or the one-hot observation of the env words) of a tile -> the three part tiles; 8 consecutive threads
// fetch the 8 chunks of one row, kSteps row steps per thread (128 threads: 8 steps of 16 rows, 256 threads: 4 of 32).
// All rows' loads are in flight before the first split: the first tile's gather sits on the launch's critical path (two
// dependent round trips: leaf parent, then the latent row).
template <bool kInitial, int kSteps>
__device__ __forceinline__ void gather_tile(const Args& a, uint8_t (*t0)[kAtomA], int tile, int gtid) {
  constexpr int kRowStep = kM / kSteps;
  const int64_t row0 = (int64_t)tile * kM, n = a.n;
  const int chunk = gtid & 7, r0 = gtid >> 3;
  if (kInitial) {  // one-hot observation: column 3 d + peg(d), columns 8 chunk .. 8 chunk + 7 of each row
    uint32_t w[kSteps];
#pragma unroll
    for (int i = 0; i < kSteps; ++i) {
      const int64_t r = row0 + r0 + kRowStep * i;
      w[i] = a.words[r < n ? r : n - 1];
    }
#pragma unroll
    for (int i = 0; i < kSteps; ++i) {
      float x[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int col = chunk * 8 + j, d = col / 3;
        x[j] = (col < 3 * a.n_disks && ((w[i] >> (2 * d)) & 3u) == (uint32_t)(col - 3 * d)) ? 1.f : 0.f;
      }
      store_parts8(t0, r0 + kRowStep * i, chunk, x);
    }
  } else {
    int64_t irow[kSteps];
#pragma unroll
    for (int i = 0; i < kSteps; ++i) {
      const int64_t r = row0 + r0 + kRowStep * i;
      const int64_t it = r < n ? r : n - 1;
      irow[i] = it * a.in_rows_per_item + (a.in_row ? (int64_t)a.in_row[it] : 0);
    }
    if (a.latent_dtype == HMZ_LATENT_F32) {
      float4 u[kSteps][2];
#pragma unroll
      for (int i = 0; i < kSteps; ++i) {
        const float4* src = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(a.lat_in) + irow[i] * kLatent + chunk * 8);
        u[i][0] = __ldcs(src);
        u[i][1] = __ldcs(src + 1);
      }
#pragma unroll
      for (int i = 0; i < kSteps; ++i) {
        const float x[8] = {u[i][0].x, u[i][0].y, u[i][0].z, u[i][0].w, u[i][1].x, u[i][1].y, u[i][1].z, u[i][1].w};
        store_parts8(t0, r0 + kRowStep * i, chunk, x);
      }
    } else {
      uint4 q[kSteps];
#pragma unroll
      for (int i = 0; i < kSteps; ++i)
        q[i] = __ldcs(reinterpret_cast<const uint4*>(reinterpret_cast<const uint16_t*>(a.lat_in) + irow[i] * kLatent + chunk * 8));
#pragma unroll
      for (int i = 0; i < kSteps; ++i) {
        const uint32_t pk[4] = {q[i].x, q[i].y, q[i].z, q[i].w};
        float x[8];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          x[2 * j] = bf_lo(pk[j]);
          x[2 * j + 1] = bf_hi(pk[j]);
        }
        store_parts8(t0, r0 + kRowStep * i, chunk, x);
      }
    }
  }
  fence_proxy_async();
}

// kInitial = false: recurrent_inference — networks dynamics, reward, value, policy; input = gathered latents.
// kInitial = true : initial_inference  — networks representation (in the dynamics network's place), value, policy;
//                   input = utils.oneHot_encoding (utils.py:9-25) of the env words (exact in bf16: only part 0 is non-zero).
template <bool kInitial>
__global__ void __launch_bounds__(kThreads, 1) net_x3(const __grid_constant__ Args a) {
  extern __shared__ uint8_t smem_raw[];
  Smem& s = *reinterpret_cast<Smem*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int tid = threadIdx.x, warp = tid >> 5;
  const int split = (!kInitial && a.head_split == 3) ? 3 : 1;
  const int role = split == 3 ? (int)blockIdx.x % 3 : -1;  // -1: every network
  const int cta = (int)blockIdx.x / split, n_cta = (int)gridDim.x / split;
  const int n_steps = kInitial ? 12 : (split == 3 ? 8 : 16);  // chunks per tile in this CTA
  // chunk gi of this CTA -> chunk g = 4 network + c of the pass order dynamics, reward, value, policy
  auto chunk_of = [&](int gi) {
    if (kInitial) return gi < 4 ? gi : gi + 4;  // no reward head at the root
    return (split == 1 || gi < 4) ? gi : (role + 1) * 4 + (gi - 4);
  };
  const int n_tiles = a.n_tiles;
  const int64_t n = a.n;
  bool tl_on = a.timeline != 0 && blockIdx.x == 0 && (tid & 31) == 0;  // (switched off after the first tile)
  if (tid == 0) X3_TL(110);

  if (tid == 32) {
    for (int j = 0; j < 2; ++j) {
      mbar_init(&s.bar_w1full[j], 1);
      mbar_init(&s.bar_w1free[j], 1);
      mbar_init(&s.bar_w2full[j], 1);
      mbar_init(&s.bar_w2free[j], 1);
    }
    for (int j = 0; j < (int)kBufs; ++j) {
      mbar_init(&s.bar_d[j], 1);
      mbar_init(&s.bar_a[j], kEpiThreads);
      mbar_init(&s.bar_hfree[j], 1);
    }
    mbar_init(&s.bar_g, kOutThreads);
    mbar_init(&s.bar_g0, kEpiThreads + kOutThreads);
    mbar_init(&s.bar_o, 1);
    mbar_init(&s.bar_out, kOutThreads);
    mbar_init(&s.bar_raw, kOutThreads);
    mbar_init(&s.bar_hn, kOutThreads);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&s.tmem_base)), "r"(512u)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = s.tmem_base;
  if (tid == 0) X3_TL(111);

  if (warp == kLoaderWarp) {
    // ================================= loader warp =================================
    // First-layer blocks run one chunk ahead of second-layer blocks (W1(0), W1(1), W2(0), W1(2), W2(1), ...): a first-layer
    // slot frees as soon as the first layer two chunks back has completed, a second-layer slot only when that chunk's
    // second layer has — queued strictly in chunk order, the next first-layer block would sit behind that later event.
    const uint32_t total = cta < n_tiles ? (uint32_t)((n_tiles - cta + n_cta - 1) / n_cta) * (uint32_t)n_steps : 0u;
    auto load = [&](uint32_t G, bool second) {  // chunk counter of this CTA: slot G & 1, use G >> 1
      const int g = chunk_of((int)(G % (uint32_t)n_steps));
      const uint32_t slot = G & 1u, use = G >> 1;
      const uint8_t* wsec = a.wsec;
      if (a.block_set != nullptr) {  // the tile this chunk belongs to: the CTA's (G / n_steps)-th
        const int tile = cta + (int)(G / (uint32_t)n_steps) * n_cta;
        wsec += (int64_t)a.block_set[tile >> 1] * a.weight_stride;
      }
      const uint8_t* blk = wsec + (size_t)((kInitial && g < 4) ? kRepBlock0 + g : g) * kBlockStride;
      if (!second) {
        if (use >= 1u) mbar_wait(&s.bar_w1free[slot], (use - 1u) & 1u);
        if (G < (uint32_t)n_steps) X3_TL(128 + g);
        if (elect_one()) tma_load(s.w1[slot], blk, kW1Bytes, &s.bar_w1full[slot]);
      } else {
        if (use >= 1u) mbar_wait(&s.bar_w2free[slot], (use - 1u) & 1u);
        if (elect_one()) tma_load(s.w2[slot], blk + kSlot, 3u * n2_of(g >> 2) * 160u, &s.bar_w2full[slot]);
      }
      __syncwarp();
    };
    for (uint32_t j = 0; j <= total; ++j) {
      if (j < total) load(j, false);
      if (j >= 1u) load(j - 1u, true);
    }
  } else if (warp == kMma1Warp || warp == kMma1bWarp) {
    // ========================= first-layer issuing warps =========================
    // (two of them, one for the even and one for the odd chunks of the CTA's chunk sequence — each always uses the same
    // weight slot: between two chunks a warp spends ~800 clk in its barrier waits and fences, which the other warp's
    // issue now covers; the timeline showed the single first-layer warp's loop, not the tensor pipe, pacing the kernel)
    const uint32_t my_parity = warp == kMma1Warp ? 0u : 1u;
    // Two issuing warps, one per layer kind: issuing a tcgen05.mma blocks for about its execution time, so a single warp
    // would serialise the second layer of chunk g behind the issue of the first layer of chunk g + 1 (and behind its own
    // waits); the tensor core takes the two streams in arrival order.  The write-after-read hazard on an accumulator
    // buffer — the first layer of chunk G + 2 overwrites what the second layer of chunk G reads as its A operand —
    // is then ordered by an mbarrier (bar_hfree: second layer of chunk G complete) instead of by issue order.
    const uint32_t id128 = umma_idesc(128), id64 = umma_idesc(64);
    const uint32_t ax = smem_u32(s.ax);
    uint32_t G = 0, ph_tile = 0;
    for (int tile = cta; tile < n_tiles; tile += n_cta) {
#pragma unroll 1
      for (int gi = 0; gi < n_steps; ++gi, ++G) {
        if ((G & 1u) != my_parity) continue;
        const int g = chunk_of(gi);
        const uint32_t slot = G & 1u, use = G >> 1, buf = G % kBufs, bu = G / kBufs;
        X3_TL(112 + g);
        mbar_wait(&s.bar_w1full[slot], use & 1u);
        X3_TL(144 + g);
        if (bu >= 1u) mbar_wait(&s.bar_hfree[buf], (bu - 1u) & 1u);  // accumulator buffer no longer read
        // this chunk's A tile (each issuing warp checks for itself: the other one may have done the network's first chunk)
        if (g < 4) {                                     // input tile gathered
          if (tile == cta) mbar_wait(&s.bar_g0, 0u);
          else mbar_wait(&s.bar_g, ph_tile ^ 1u);        // (bar_g's first phase belongs to the CTA's second tile)
        }
        else if (g < 8) mbar_wait(&s.bar_raw, ph_tile);  // raw latent tile written (reward head input)
        else mbar_wait(&s.bar_hn, ph_tile);              // normalised latent tile written (value / policy head input)
        tc_fence_after();
        X3_TL(g);
        if (elect_one()) {
          const uint32_t D1 = tmem + 128u * buf;
          const uint32_t w = smem_u32(s.w1[slot]);
          const uint64_t b01 = desc_sw128(w), b2 = desc_sw128(w + 128u * 128u);
          if ((g >> 2) <= 1) {  // dynamics / representation (input tile), reward head (raw latent tile): A from shared memory
            const uint32_t a_in = smem_u32(s.t0[0]);
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
#pragma unroll
              for (int i = 0; i < 3; ++i)
                umma(D1, desc_sw128(a_in + (uint32_t)i * kAtomA) + (uint64_t)(kk * 2), b01 + (uint64_t)(kk * 2), id128, (kk | i) ? 1u : 0u);
              umma(D1 + 64u, desc_sw128(a_in) + (uint64_t)(kk * 2), b2 + (uint64_t)(kk * 2), id64, 1u);
            }
          } else {  // value / policy heads: the normalised latent's parts are a TMEM operand (no shared-memory reads for A:
                    // a first layer with both operands in shared memory runs at the port's 128 B/clk)
            const uint32_t hn = tmem + kColHn;
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
#pragma unroll
              for (int i = 0; i < 3; ++i)
                umma_ts(D1, hn + 32u * (uint32_t)i + 8u * (uint32_t)kk, b01 + (uint64_t)(kk * 2), id128, (kk | i) ? 1u : 0u);
              umma_ts(D1 + 64u, hn + 8u * (uint32_t)kk, b2 + (uint64_t)(kk * 2), id64, 1u);
            }
          }
          umma(D1, desc_plain(ax), desc_plain(w + kW1Main), id128, 1u);
          umma(D1 + 64u, desc_plain(ax), desc_plain(w + kW1Main + plain_off(128, 0)), id64, 1u);
          umma_commit(&s.bar_d[buf]);
          umma_commit(&s.bar_w1free[slot]);
        }
        __syncwarp();
        X3_TL(16 + g);
      }
      ph_tile ^= 1u;
      tl_on = false;
    }
  } else if (warp == kMma2Warp) {
    // ========================= second-layer issuing warp =========================
    // the chunk's K = 64 slice, A = the three hidden parts in TMEM
    const uint32_t ax = smem_u32(s.ax);
    uint32_t G = 0, ph_tile = 0, ph_out = 0;
    bool first_tile = true;
    for (int tile = cta; tile < n_tiles; tile += n_cta) {
#pragma unroll 1
      for (int gi = 0; gi < n_steps; ++gi, ++G) {
        const int g = chunk_of(gi);
        const uint32_t slot = G & 1u, use = G >> 1, buf = G % kBufs, bu = G / kBufs;
        const int net = g >> 2, c = g & 3;
        mbar_wait(&s.bar_w2full[slot], use & 1u);
        mbar_wait(&s.bar_a[buf], bu & 1u);
        // D2 must have been drained by the output epilogue of the network this CTA ran before: the dynamics network's
        // (bar_raw) for the network that follows it, a head's (bar_out) otherwise
        if (gi == 4) mbar_wait(&s.bar_raw, ph_tile);
        if (c == 0 && gi != 4 && (gi != 0 || !first_tile)) {
          mbar_wait(&s.bar_out, ph_out);
          ph_out ^= 1u;
        }
        tc_fence_after();
        X3_TL(32 + g);
        if (elect_one()) {
          const uint32_t n2 = n2_of(net);
          const uint32_t ida = umma_idesc(2u * n2), idb = umma_idesc(n2);
          const uint32_t D1 = tmem + 128u * buf, D2 = tmem + kColD2;
          const uint32_t w = smem_u32(s.w2[slot]);
          const uint64_t b01 = desc_sw128(w), b2 = desc_sw128(w + 2u * n2 * 128u);
          if (c == 0) {  // bias step clears D2
            umma(D2, desc_plain(ax), desc_plain(w + 3u * n2 * 128u), ida, 0u);
            umma(D2 + n2, desc_plain(ax), desc_plain(w + 3u * n2 * 128u + plain_off((int)(2u * n2), 0)), idb, 1u);
          }
#pragma unroll
          for (int b4 = 0; b4 < 4; ++b4) {
            const uint32_t h0 = D1 + 16u * b4, h1 = h0 + 8u, h2 = h0 + 64u;
            umma_ts(D2, h0, b01 + (uint64_t)(b4 * 2), ida, 1u);
            umma_ts(D2, h1, b01 + (uint64_t)(b4 * 2), ida, 1u);
            umma_ts(D2, h2, b01 + (uint64_t)(b4 * 2), ida, 1u);
            umma_ts(D2 + n2, h0, b2 + (uint64_t)(b4 * 2), idb, 1u);
          }
          if (c == 3) umma_commit(&s.bar_o);
          umma_commit(&s.bar_w2free[slot]);
          umma_commit(&s.bar_hfree[buf]);
        }
        __syncwarp();
        X3_TL(48 + g);
      }
      ph_tile ^= 1u;
      first_tile = false;
      tl_on = false;
    }
  } else if (warp < kOutWarp0) {
    // ================================= hidden-epilogue warps =================================
    const int quarter = warp & 3, half = warp >> 2;
    const uint32_t T = tmem + ((uint32_t)(quarter * 32) << 16);
    uint32_t G = 0;
    tl_on = tl_on && tid == 0;
    if (cta < n_tiles) {  // these warps have nothing to do until the first chunk's accumulator: they gather the first tile
      X3_TL(104);
      gather_tile<kInitial, 4>(a, s.t0, cta, tid);
      mbar_arrive(&s.bar_g0);
      X3_TL(105);
    }
    for (int tile = cta; tile < n_tiles; tile += n_cta) {
#pragma unroll 1
      for (int gi = 0; gi < n_steps; ++gi, ++G) {
        const int g = chunk_of(gi);
        const uint32_t buf = G % kBufs, bu = G / kBufs;
        mbar_wait(&s.bar_d[buf], bu & 1u);
        tc_fence_after();
        X3_TL(64 + g);
        hidden_epilogue(T + 128u * buf, half);
        tc_fence_before();
        mbar_arrive(&s.bar_a[buf]);
        X3_TL(80 + g);
      }
      tl_on = false;
    }
  } else {
    // ================================= output warps =================================
    // Four warps, thread = row: the gather of a tile's input, the new latent (raw -> reward head, normalised -> value /
    // policy heads and HBM) and the heads' outputs — apart from the eight hidden-epilogue warps, so that the chunk
    // epilogues of the next network never wait behind an output epilogue.  The NEXT tile's input is gathered right
    // after the reward head (the last reader of the raw-latent tile) while the value / policy heads still run.
    const int otid = tid - kOutWarp0 * 32;
    const int row = otid;  // = TMEM lane: warp & 3 is the lane quarter
    const uint32_t D2 = tmem + ((uint32_t)((warp & 3) * 32) << 16) + kColD2;
    uint32_t ph_o = 0;
    tl_on = tl_on && otid == 0;
    auto gather = [&](int tile) { gather_tile<kInitial, 8>(a, s.t0, tile, otid); };
    // extra A slice of this row: one-hot(action) at k = 0..5, the constant 1 at k = 6; then the tile is handed over
    auto publish_inputs = [&](int tile, uint64_t* bar) {
      const int64_t it = ((int64_t)tile * kM + row) < n ? ((int64_t)tile * kM + row) : n - 1;
      const uint32_t act = kInitial ? 0u : min((uint32_t)a.actions[it], (uint32_t)(kActions - 1));
      const uint32_t one = kInitial ? 0u : 0x3F80u << ((act & 1u) * 16u);
      const uint32_t ax = smem_u32(s.ax);
      asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(ax + plain_off(row, 0)), "r"((act >> 1) == 0u ? one : 0u),
                   "r"((act >> 1) == 1u ? one : 0u), "r"((act >> 1) == 2u ? one : 0u), "r"(0x3F80u)
                   : "memory");
      asm volatile("st.shared.v4.u32 [%0], {%1, %1, %1, %1};" ::"r"(ax + plain_off(row, 1)), "r"(0u) : "memory");
      fence_proxy_async();
      mbar_arrive(bar);
    };
    if (cta < n_tiles) publish_inputs(cta, &s.bar_g0);
    for (int tile = cta; tile < n_tiles; tile += n_cta) {
      const int64_t item = (int64_t)tile * kM + row;
      const int next_tile = tile + n_cta;
#pragma unroll 1
      for (int net = 0; net < 4; ++net) {  // dynamics, reward, value, policy
        if (split == 3 && net != 0 && net != role + 1) continue;
        if (kInitial && net == 1) continue;
        const bool last_net = split == 3 ? net != 0 : net == 3;
        // the raw-latent tile has no reader left in this CTA
        const bool raw_tile_free = kInitial ? net == 0 : (split == 3 ? net != 0 : net == 1);
        mbar_wait(&s.bar_o, ph_o);
        ph_o ^= 1u;
        tc_fence_after();
        X3_TL(96 + net);
        if (net == 0) {
          // ---- new latent.  The raw latent feeds the reward head: publish it first so that head's first layers overlap
          // the normalisation.
          float raw[64];
#pragma unroll
          for (int j = 0; j < 4; ++j) ld_sum16(D2 + 16 * j, D2 + 64 + 16 * j, *reinterpret_cast<float(*)[16]>(&raw[16 * j]));
          tc_fence_before();
          if (!kInitial) {
#pragma unroll
            for (int c = 0; c < 8; ++c) store_parts8(s.t0, row, c, *reinterpret_cast<float(*)[8]>(&raw[c * 8]));
            fence_proxy_async();
          }
          mbar_arrive(&s.bar_raw);
          X3_TL(106);
          float mn4[4], mx4[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) mn4[i] = mx4[i] = raw[i];
#pragma unroll
          for (int i = 4; i < 64; ++i) {
            mn4[i & 3] = fminf(mn4[i & 3], raw[i]);
            mx4[i & 3] = fmaxf(mx4[i & 3], raw[i]);
          }
          const float mn = fminf(fminf(mn4[0], mn4[1]), fminf(mn4[2], mn4[3]));
          const float mx = fmaxf(fmaxf(mx4[0], mx4[1]), fmaxf(mx4[2], mx4[3]));
          // normalize_h_state (networks.py:191-196); the quotient as a product with the correctly rounded reciprocal
          // (<= 1.5 ulp from the division, far inside the gate)
          const float inv = __frcp_rn(__fadd_rn(__fsub_rn(mx, mn), 1e-8f));
          const int64_t orow = item * a.out_rows_per_item + a.out_row;
#pragma unroll
          for (int c = 0; c < 8; ++c) {
            float hn[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) hn[j] = __fmul_rn(__fsub_rn(raw[c * 8 + j], mn), inv);
            {  // three bf16 parts of the eight values -> four packed columns per part (lane = row, one column = two k)
              uint32_t pp[3][4];
#pragma unroll
              for (int j = 0; j < 4; ++j) split3(hn[2 * j], hn[2 * j + 1], pp[0][j], pp[1][j], pp[2][j]);
#pragma unroll
              for (int i = 0; i < 3; ++i) tmem_st4(D2 - kColD2 + kColHn + 32u * (uint32_t)i + 4u * (uint32_t)c, pp[i]);
            }
            if (item < n && role <= 0) {  // (head split: the reward CTA stores the rows)
              if (a.latent_dtype == HMZ_LATENT_F32) {
                float4* dst = reinterpret_cast<float4*>(reinterpret_cast<float*>(a.lat_out) + orow * kLatent + c * 8);
                __stcs(dst, make_float4(hn[0], hn[1], hn[2], hn[3]));
                __stcs(dst + 1, make_float4(hn[4], hn[5], hn[6], hn[7]));
              } else {
                __stcs(reinterpret_cast<uint4*>(reinterpret_cast<uint16_t*>(a.lat_out) + orow * kLatent + c * 8),
                       make_uint4(pack_bf16(hn[0], hn[1]), pack_bf16(hn[2], hn[3]), pack_bf16(hn[4], hn[5]), pack_bf16(hn[6], hn[7])));
              }
            }
          }
          tmem_st_wait();
          tc_fence_before();
          mbar_arrive(&s.bar_hn);
        } else if (net == 3) {  // F.softmax(pi_logits) (networks.py:109)
          float lg[16];
          ld_sum16(D2, D2 + 16, lg);
          tc_fence_before();
          mbar_arrive(&s.bar_out);
          float mx = lg[0], den = 0.f;
#pragma unroll
          for (int k = 1; k < kActions; ++k) mx = fmaxf(mx, lg[k]);
#pragma unroll
          for (int k = 0; k < kActions; ++k) {
            lg[k] = expf(lg[k] - mx);
            den += lg[k];
          }
          if (item < n) {
#pragma unroll
            for (int k = 0; k < kActions; ++k) a.p_out[item * kActions + k] = __fdiv_rn(lg[k], den);
          }
        } else {  // support transform (networks.py:152-189) of the 33 logits
          float lg[48];
#pragma unroll
          for (int j = 0; j < 3; ++j) ld_sum16(D2 + 16 * j, D2 + 48 + 16 * j, *reinterpret_cast<float(*)[16]>(&lg[16 * j]));
          tc_fence_before();
          mbar_arrive(&s.bar_out);
          const float x = support_to_scalar([&](int i) { return lg[i]; });
          if (item < n) (net == 1 ? a.r_out : a.v_out)[item] = x;
        }
        if (next_tile < n_tiles) {
          // the reward head's first layers were the last readers of the raw-latent tile: gather the next tile into it;
          // after the last network every tcgen05.mma of the tile has completed and the extra A slice may change hands
          if (raw_tile_free) gather(next_tile);
          if (last_net) publish_inputs(next_tile, &s.bar_g);
        }
        X3_TL(100 + net);
      }
      tl_on = false;
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512u) : "memory");
  }
}

// ---- host-side packing ----------------------------------------------------------------
static uint16_t f2bf(float f) {
  uint32_t u;
  std::memcpy(&u, &f, 4);
  if ((u & 0x7FFFFFFFu) > 0x7F800000u) return (uint16_t)((u >> 16) | 0x40u);
  return (uint16_t)((u + 0x7FFFu + ((u >> 16) & 1u)) >> 16);
}
static float bf2f(uint16_t h) {
  const uint32_t u = (uint32_t)h << 16;
  float f;
  std::memcpy(&f, &u, 4);
  return f;
}
static uint16_t part_of(float w, int part) {
  uint16_t h = f2bf(w);
  for (int p = 0; p < part; ++p) {
    w = w - bf2f(h);  // exact: the residual of a bf16 rounding fits float32
    h = f2bf(w);
  }
  return h;
}
// rows [part * n_rows + r] of one SWIZZLE_128B K-atom (K = 64) followed by the extra K = 16 slice; get(r, k) is the
// float32 weight of output row r and input column k (k < 64 main, 64 + j = column j of the extra slice), 0 when absent
template <typename F>
static void pack_block(uint8_t* dst, int n_rows, F get) {
  const int rows = 3 * n_rows;
  for (int part = 0; part < 3; ++part)
    for (int r = 0; r < n_rows; ++r) {
      const int row = part * n_rows + r;
      for (int k = 0; k < 64; ++k)
        *reinterpret_cast<uint16_t*>(dst + (size_t)row * 128 + (((k >> 3) ^ (row & 7)) << 4) + (k & 7) * 2) = part_of(get(r, k), part);
      for (int k = 0; k < 16; ++k)
        *reinterpret_cast<uint16_t*>(dst + (size_t)rows * 128 + plain_off(row, k >> 3) + (k & 7) * 2) = part_of(get(r, 64 + k), part);
    }
}

int64_t fp32_offset_bytes() { return (int64_t)kSectionBytes; }
int64_t packed_bytes(int n_disks) { return fp32_offset_bytes() + (int64_t)Fp32Layout::total(n_disks) * 4; }

void pack(const float* const* t, int n_disks, void* out) {
  std::memset(out, 0, (size_t)packed_bytes(n_disks));
  // float observations (drop-in B = 1 views, arbitrary input vectors) run the FFMA kernel on the float32 copy behind the section
  pack_fp32(t, n_disks, (float*)((uint8_t*)out + fp32_offset_bytes()));
  uint8_t* sec = (uint8_t*)out;
  // state_dict order: rep(0-3) dyn(4-7) rwd(8-11) pol(12-15) val(16-19), each {w1, b1, w2, b2}; pass order dyn, rwd, val, pol
  const int first[4] = {4, 8, 16, 12};
  const int out2[4] = {kLatent, kSupport, kSupport, kActions};
  for (int net = 0; net < 4; ++net) {
    const float *w1 = t[first[net]], *b1 = t[first[net] + 1], *w2 = t[first[net] + 2], *b2 = t[first[net] + 3];
    const int in1 = net == 0 ? kLatent + kActions : kLatent;
    const int n2 = (int)n2_of(net);
    for (int c = 0; c < 4; ++c) {
      uint8_t* blk = sec + (size_t)(net * 4 + c) * kBlockStride;
      pack_block(blk, 64, [&](int r, int k) -> float {
        const int unit = 64 * c + r;
        if (k < 64) return w1[(size_t)unit * in1 + k];
        const int j = k - 64;
        if (net == 0 && j < kActions) return w1[(size_t)unit * in1 + kLatent + j];
        return j == kBiasK ? b1[unit] : 0.f;
      });
      pack_block(blk + kSlot, n2, [&](int r, int k) -> float {
        if (r >= out2[net]) return 0.f;
        if (k < 64) return w2[(size_t)r * kHidden + 64 * c + k];
        return (c == 0 && k - 64 == kBiasK) ? b2[r] : 0.f;
      });
    }
  }
  // representation_net (root inference): Linear(3N, 256) on the one-hot observation padded to K = 64, Linear(256, 64)
  const int d_in = 3 * n_disks;
  for (int c = 0; c < 4; ++c) {
    uint8_t* blk = sec + (size_t)(kRepBlock0 + c) * kBlockStride;
    pack_block(blk, 64, [&](int r, int k) -> float {
      const int unit = 64 * c + r;
      if (k < 64) return k < d_in ? t[0][(size_t)unit * d_in + k] : 0.f;
      return k - 64 == kBiasK ? t[1][unit] : 0.f;
    });
    pack_block(blk + kSlot, 64, [&](int r, int k) -> float {
      if (k < 64) return t[2][(size_t)r * kHidden + 64 * c + k];
      return (c == 0 && k - 64 == kBiasK) ? t[3][r] : 0.f;
    });
  }
}

static int prepare(int* smem_bytes) {
  static thread_local int done_dev = -1;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return fail(HMZ_ERR_CUDA, "cudaGetDevice failed (no CUDA device?)");
  *smem_bytes = (int)sizeof(Smem) + 1024;
  if (done_dev != dev) {
    cudaError_t e = cudaFuncSetAttribute(net_x3<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, *smem_bytes);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(net_x3<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, *smem_bytes);
    if (e != cudaSuccess) return fail(HMZ_ERR_CUDA, "cudaFuncSetAttribute(net_x3): %s", cudaGetErrorString(e));
    done_dev = dev;
  }
  return HMZ_OK;
}

int net_recurrent(const void* weights, const void* lat_in, int64_t in_rows_per_item, const uint16_t* in_row,
                  const uint8_t* actions, void* lat_out, int64_t out_rows_per_item, int64_t out_row, int latent_dtype,
                  float* r, float* p, float* v, int64_t n, cudaStream_t stream, const uint16_t* block_set, int64_t weight_stride,
                  bool allow_head_split) {
  int smem = 0;
  if (int rc = prepare(&smem)) return rc;
  Args a{};
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
  a.n_tiles = (int)((n + kM - 1) / kM);
  const int sms = sm_count();
  // small batches: three CTAs per tile, one head each
  a.head_split = (allow_head_split && 3 * a.n_tiles <= sms) ? 3 : 1;
  static const int tl = getenv("HMZ_X3_TIMELINE") ? atoi(getenv("HMZ_X3_TIMELINE")) : 0;
  a.timeline = tl;
  const unsigned grid = a.head_split == 3 ? 3u * (unsigned)a.n_tiles : (unsigned)(a.n_tiles < sms ? a.n_tiles : sms);
  net_x3<false><<<grid, kThreads, (size_t)smem, stream>>>(a);
  return check_launch("net_x3<recurrent>");
}

int net_initial(const void* weights, int n_disks, const uint32_t* words, void* lat_out, int64_t out_rows_per_item,
                int latent_dtype, float* p0, float* v0, int64_t n, cudaStream_t stream, const uint16_t* block_set, int64_t weight_stride) {
  int smem = 0;
  if (int rc = prepare(&smem)) return rc;
  Args a{};
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
  a.n_tiles = (int)((n + kM - 1) / kM);
  a.head_split = 1;
  const int sms = sm_count();
  net_x3<true><<<(unsigned)(a.n_tiles < sms ? a.n_tiles : sms), kThreads, (size_t)smem, stream>>>(a);
  return check_launch("net_x3<initial>");
}

int debug_read_timeline(unsigned long long* host_out) {
  return cudaMemcpyFromSymbol(host_out, g_x3_timeline, sizeof(g_x3_timeline)) == cudaSuccess ? HMZ_OK : HMZ_ERR_CUDA;
}

}  // namespace x3
}  // namespace hmz
