// Device side of the tensor-core MuZeroNet inference (hmz_net_tc.cu): PTX wrappers, shared-memory layout and the
// body of the v4 kernel as a device function, so that the stand-alone kernels (net_tc<recurrent / initial>, one launch
// per simulation) and the MLP role of the persistent search kernel (hmz_persist.cu) run the SAME code.
#pragma once
#include "hmz_net.cuh"

namespace hmz {

namespace tc {
constexpr int kM = 128;          // rows per CTA / UMMA M
constexpr uint32_t kAtomA = kM * 128;  // one K-atom (64 bf16) of a 128-row A tile: 16 KB

// A weight matrix [n_out][K] is stored as K/64 SWIZZLE_128B K-atoms of [n_out][128 B] followed by the
// "extra" K = 16 slice [n_out][32 B] in the un-swizzled core-matrix layout (8 rows x 16 B contiguous,
// the two K-chunks 128 B apart, 8-row groups 256 B apart) carrying the bias at k = 6 (and, for
// dynamic_net.0, the six one-hot action columns at k = 0..5).
constexpr uint32_t w_bytes(uint32_t n_out, uint32_t k_atoms) { return n_out * 128 * k_atoms + n_out * 32; }
constexpr uint32_t kBytesW1 = w_bytes(256, 1);   // 40960
constexpr uint32_t kBytesWg2 = w_bytes(64, 4);   // 34816
constexpr uint32_t kBytesW48 = w_bytes(48, 4);   // 26112
constexpr uint32_t kBytesW16 = w_bytes(16, 4);   // 8704
constexpr uint32_t kBytesWs1 = (kBytesW48 + 1023) / 1024 * 1024;  // second-layer slot 1 holds at most a 48-row block
// byte offsets inside the tensor-core section of the weight blob (all multiples of 1024)
constexpr uint32_t kWg1 = 0, kWg2 = 40960, kWr1 = 75776, kWr2 = 116736, kWp1 = 142848 + 1024 - 512, kWp2 = kWp1 + 40960,
                   kWv1 = kWp2 + 9216, kWv2 = kWv1 + 40960, kWh1 = kWv2 + 26112 + 512, kWh2 = kWh1 + 40960,
                   kSectionBytes = kWh2 + 34816;  // kWh*: representation_net (root inference)
static_assert(kWg2 % 1024 == 0 && kWr1 % 1024 == 0 && kWr2 % 1024 == 0 && kWp1 % 1024 == 0 && kWp2 % 1024 == 0 &&
                  kWv1 % 1024 == 0 && kWv2 % 1024 == 0 && kWh1 % 1024 == 0 && kWh2 % 1024 == 0,
              "weight blocks must be 1024-byte aligned for SWIZZLE_128B");
static_assert(kWr1 >= kWg2 + kBytesWg2 && kWr2 >= kWr1 + kBytesW1 && kWp1 >= kWr2 + kBytesW48 && kWp2 >= kWp1 + kBytesW1 &&
                  kWv1 >= kWp2 + kBytesW16 && kWv2 >= kWv1 + kBytesW1,
              "weight blocks overlap");
constexpr int kBiasK = 6;  // column of the extra slice that multiplies the constant 1

// Debug timeline: block 0 records clock64() at phase boundaries when HMZ_TC_TIMELINE=1 (tools only).
static __device__ unsigned long long g_timeline[96];

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ unsigned long long globaltimer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
constexpr unsigned long long kWaitTimeoutNs = 20ull * 1000ull * 1000ull * 1000ull;
// A wait that has lasted 20 s is a protocol failure: trap (the launch fails with an error) rather than hang the GPU.
// The clock is read once every 2^16 polls, so a wait that succeeds pays nothing for the guard.
struct WaitGuard {
  uint32_t spins = 0;
  unsigned long long t0 = 0;
  bool expired = false;  // HMZ_WATCHDOG_SOFT (tooling build): the wait gives up after 2 s instead of trapping, so that the
                         // kernels end and the caller of the wait can report what it was waiting for
  __device__ __forceinline__ void poll() {
    if ((++spins & 0xFFFFu) == 0u) {
      const unsigned long long now = globaltimer_ns();
      if (t0 == 0) t0 = now;
#ifdef HMZ_WATCHDOG_SOFT
      else if (now - t0 > 2000000000ull) expired = true;
#else
      else if (now - t0 > kWaitTimeoutNs) __trap();
#endif
    }
  }
};
// (Intra-CTA waits stay an unguarded try_wait loop: a guard costs registers in every wait of the hot kernel; the waits
// that depend on OTHER CTAs — the hand-offs of the persistent kernel, which everything else waits behind — are guarded.)
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t"
      "}" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
// 1-D TMA bulk copy global -> shared, completion signalled on an mbarrier (SASS: UBLKCP)
__device__ __forceinline__ void tma_load(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  mbar_expect_tx(bar, bytes);
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
// One lane of a fully converged warp (the control warp runs warp-uniform code and elects a lane only
// around the instructions that must be issued once: descriptors then stay in uniform registers
// instead of being moved there with R2UR before every tcgen05.mma).
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// Shared-memory matrix descriptors (cute::UMMA::SmemDescriptor, sm100; version field = 1).
// K-major SWIZZLE_128B: LBO unused (1), SBO = 1024 B between 8-row groups, layout type 2.
__device__ __forceinline__ uint64_t desc_sw128(uint32_t smem_addr) {
  const uint64_t hi = 64ull | (1ull << 14) | (2ull << 29);
  return (uint64_t)(((smem_addr >> 4) & 0x3FFFu) | (1u << 16)) | (hi << 32);
}
// K-major, no swizzle (core matrices of 8 rows x 16 B): LBO = 128 B between the two K-chunks,
// SBO = 256 B between 8-row groups, layout type 0.
__device__ __forceinline__ uint64_t desc_plain(uint32_t smem_addr) {
  const uint64_t hi = 16ull | (1ull << 14);
  return (uint64_t)(((smem_addr >> 4) & 0x3FFFu) | (8u << 16)) | (hi << 32);
}
// byte offset of (row, 16-byte chunk c in {0, 1}) inside a core-matrix-layout K = 16 slice
__device__ __host__ __forceinline__ uint32_t plain_off(int row, int c) { return (uint32_t)((row >> 3) * 256 + c * 128 + (row & 7) * 16); }

// kind::f16 instruction descriptor: D = f32, A = B = bf16, both K-major, M = 128, N = n
__device__ __forceinline__ uint32_t umma_idesc(uint32_t n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((n >> 3) << 17) | ((128u >> 4) << 24);
}
__device__ __forceinline__ void umma(uint32_t tmem_d, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// 32 lanes x 32 consecutive columns of TMEM -> 32 registers per thread (thread = lane = row).
// Issue and wait are separate so that the next chunk's load overlaps the current chunk's math; the
// wait names the destination registers as in/out operands so no use can be scheduled above it.
__device__ __forceinline__ void tmem_ld32_issue(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait(uint32_t (&r)[32]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]),
                 "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]), "+r"(r[16]),
                 "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]), "+r"(r[24]),
                 "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31])
               :
               : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
  uint32_t r[32];
  tmem_ld32_issue(taddr, r);
  tmem_ld_wait(r);
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]),
                 "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15])
               :
               : "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
// relu + round-to-nearest-even bf16 of two floats in one conversion
__device__ __forceinline__ uint32_t pack_relu_bf16(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
// 16-byte chunk `chunk` (8 bf16) of row `row` inside a [rows][128 B] SWIZZLE_128B K-atom
__device__ __forceinline__ uint32_t sw128(int row, int chunk) { return (uint32_t)(row * 128 + ((chunk ^ (row & 7)) << 4)); }

// =====================================================================================
// net_tc (v4): two 128-search tiles per CTA pass, ping-ponged.
//
//   * Both tiles consume every weight block from the same shared-memory copy (double-buffered
//     per layer kind, streamed by a dedicated loader warp), which halves the L2 -> SM weight
//     traffic per search, and the tensor core works on one tile while the other tile's epilogue
//     warps drain TMEM.
//   * Hidden activations never touch shared memory: the epilogue reads the float32 accumulator
//     with tcgen05.ld, applies relu + bf16 and writes the packed row back IN PLACE with
//     tcgen05.st; the second-layer MMA takes its A operand from TMEM (the .ts form of
//     tcgen05.mma).  TMEM columns of tile t (base 256 t):
//         [0,128)   H0: first-layer accumulator, hidden units 0..127  -> A1 k 0..127 in [0,64)
//         [64,128)  O : second-layer accumulator (free once H0 is drained)
//         [128,256) H1: hidden units 128..255                         -> A1 k 128..255 in [128,192)
//   * The kernel is persistent over tile pairs (grid = min(pairs, SMs)).
//
// 22 warps: 2 x 8 hidden-epilogue warps (warp -> TMEM lane quarter w & 3, column half (w >> 2) & 1),
// 4 output warps shared by both tiles, one MMA-issuing warp, one loader warp.
namespace v4 {
constexpr int kHidThreadsPerTile = 256;
constexpr int kSmallWarp0 = 16, kMmaWarp = 20, kLoaderWarp = 21, kMmaWarp1 = 22;  // one MMA-issuing warp per tile
constexpr int kThreads = 23 * 32;
constexpr int kLaunchThreads = kThreads;
constexpr uint32_t kColsPerTile = 256, kColH1 = 128, kColO = 64;

struct __align__(1024) Tile {
  uint8_t a0[kAtomA];   // input latent tile, later the raw (un-normalised) new latent
  uint8_t ahn[kAtomA];  // normalised new latent
  uint8_t ax[kM * 32];  // extra A slice [onehot(action) (6), 1, 0 x 9] per row, core-matrix layout
};
struct __align__(1024) Smem {
  Tile t[2];
  uint8_t wf[2][kBytesW1];   // first-layer weight blocks (+ extra slice), double-buffered: slot = network & 1
  uint8_t ws0[kBytesWg2];    // second-layer weight blocks (+ extra slice), slot 0: dynamics / representation, value
  uint8_t ws1[kBytesWs1];    // slot 1: reward, policy (the smaller blocks: leaves room for a tree block's tables on the SM)
  float2 row_minmax[2][2][kM];
  uint64_t bar_wfull[2][2];  // [kind][slot] TMA landed
  uint64_t bar_wfree[2][2];  // [kind][slot] both tiles' MMAs reading the slot have completed
  uint64_t bar_g[2];         // gather done: A0 and AX of the tile written (384 arrivals)
  uint64_t bar_d[2];         // [tile] first-layer accumulator complete
  uint64_t bar_a[2];         // [tile] A1 written back to TMEM (256 arrivals)
  uint64_t bar_o[2];         // dynamics second layer complete (raw latent in O)
  uint64_t bar_s[2];         // head second layer complete (logits in O)
  uint64_t bar_raw[2];       // raw latent tile written, O copied out (256 arrivals)
  uint64_t bar_hn[2];        // normalised latent tile written (256 arrivals)
  uint64_t bar_fin[2];       // head logits copied out of O (128 arrivals)
  uint64_t bar_end;          // every MMA has completed
  uint64_t bar_pass;         // persistent mode: every global store of the pass has been issued (640 arrivals)
  uint32_t tmem_base;
};

// network order of a pass: dynamics, reward, VALUE, POLICY — the policy head's output (a 6-way softmax) is the cheapest,
// so it goes last, where nothing overlaps the output warps' work
static __constant__ uint32_t c_block_off[8] = {kWg1, kWg2, kWr1, kWr2, kWv1, kWv2, kWp1, kWp2};
static __constant__ uint32_t c_block_bytes[8] = {kBytesW1, kBytesWg2, kBytesW1, kBytesW48, kBytesW1, kBytesW48, kBytesW1, kBytesW16};

// D = A x B^T with A in TMEM (lane = row, one 32-bit column = two consecutive k)
__device__ __forceinline__ void umma_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "r"(tmem_a), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tmem_ld16_issue(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld16_wait(uint32_t (&r)[16]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]),
                 "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15])
               :
               : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&r)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(r[0]),
               "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// relu + bf16 of 16 accumulator columns, written back as 8 packed columns
__device__ __forceinline__ void hidden_chunk_tmem(uint32_t dst, const uint32_t (&acc)[16]) {
  uint32_t pk[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) pk[j] = pack_relu_bf16(__uint_as_float(acc[2 * j]), __uint_as_float(acc[2 * j + 1]));
  tmem_st8(dst, pk);
}
// Hidden-layer epilogue of one column half: H[0:128) float32 -> relu -> bf16 -> A1 in H[0:64), in place.
// Chunk c (columns 16c..16c+15) lands in columns 8c..8c+7, always behind the read pointer; the TMEM
// load of chunk c+1 is in flight while chunk c is converted.  (Round 2: re-dividing the CTA's registers with setmaxnreg so that these warps could hold 32-column batches does not
// work from one function — ptxas 12.9 compiles the WHOLE kernel to the smallest setmaxnreg value it sees.)
// (tcgen05.wait::ld waits for EVERY outstanding
// load, so each chunk still exposes most of one TMEM load latency, ~170 clk; requesting 64 columns per wait
// was measured SLOWER: the 64 live registers spill under the 80-register cap of a 704-thread CTA; 32 columns
// per wait without double buffering was slower too, 30.8 vs 27.3 us per launch.  Pooling all 16 epilogue
// warps on one tile's layer at a time (4 chunks per warp, 750 clk per layer instead of ~1,400) was also tried:
// the packed activations then leave only 32-column holes, every second layer needs two accumulators and twice
// the tcgen05.mma instructions from the single issuing lane, and the latent epilogues serialise: 29.1 us.)
__device__ __forceinline__ void hidden_epilogue_tmem(uint32_t h) {
  uint32_t va[16], vb[16];
  tmem_ld16_issue(h, va);
#pragma unroll
  for (int c = 0; c < 8; c += 2) {
    tmem_ld16_wait(va);
    tmem_ld16_issue(h + 16 * (c + 1), vb);
    hidden_chunk_tmem(h + 8 * c, va);
    tmem_ld16_wait(vb);
    if (c + 2 < 8) tmem_ld16_issue(h + 16 * (c + 2), va);
    hidden_chunk_tmem(h + 8 * (c + 1), vb);
  }
  tmem_st_wait();
}

#define TL4(slot) do { if ((timeline & 1) && cta == 0 && pass == (timeline >> 8)) g_timeline[slot] = clock64(); } while (0)  // bits 8+: the traced pass

// Arguments of one network pass set (the stand-alone kernels' parameter list).
struct TcArgs {
  const uint8_t* wsec;        // tensor-core section of the weight blob
  const void* lat_in;         // input latents (recurrent)
  int64_t in_rows_per_item;
  const uint16_t* in_row;     // per-item input row (leaf_parent), nullable = 0
  const uint8_t* actions;     // per-item action (recurrent)
  const uint32_t* words;      // env words (initial)
  int n_disks;
  void* lat_out;
  int64_t out_rows_per_item, out_row;
  int latent_dtype;
  float *r_out, *p_out, *v_out;
  int64_t n;                  // items
  int n_pairs;                // tile pairs = ceil(n / 256)
  int head_split;             // 3: small batches (3 x tile pairs <= SMs) — CTAs 3 p, 3 p + 1, 3 p + 2 all run the dynamics network
                              // of pair p and then ONE head each (reward + the latent rows / value / policy): the per-simulation
                              // chain of a pass shrinks from four networks to two while idle SMs do the redundant work; else 1
  int timeline;               // tooling / PDL switches of the stand-alone kernels
  unsigned long long* gantt;  // tooling (hmz_debug_gantt), nullable
  const uint16_t* block_set;  // nullable (stand-alone kernels only): weight set of each tile pair (hmz_multi_t), at
  int64_t weight_stride;      // wsec + block_set[pair] * weight_stride
};

// Hand-off state of the persistent search kernel (hmz_persist.cu), in global memory; zeroed before every launch.
//   tree_head      ticket counter of the tree warps: ticket t = slice t % 16 of work item t / 16
//   q_tail         number of items pushed by the MLP CTAs; item index = n_pairs + position (items [0, n_pairs) are the
//                  implicit first selections of every pair)
//   tree_done[p]   (one 32-byte sector per pair) warps that have finished pair p's tree phases: 16 per simulation
//   queue[slot]    (item index + 1) << 32 | pair | sim << 16, published with a release store
struct PersistCtl {
  uint32_t* tree_head;
  uint32_t* q_tail;
  uint32_t* tree_done;  // stride 8 words
  unsigned long long* queue;
  uint32_t q_mask;      // capacity - 1 (power of two)
  int n_sims;
  unsigned long long* stats;  // tooling (HMZ_PERSIST_STATS=1), nullable: clock64 sums, see hmz_debug_persist_stats
  uint32_t* mlp_done;         // server schedule (nullable; stride 8 words): mlp_done[pair] = simulations whose network outputs are
                              // complete — the tree kernels' warps wait on it; when set, no item is pushed to the queue
  uint32_t* group_done;       // server schedule (nullable): group_done[pair / pairs_per_group] += 1 per finished pass (release): the
                              // stream of the group's tree launches waits on it (cuStreamWaitValue32)
  int pairs_per_group;
  int rotate;                 // 1: a CTA's residue class of tile pairs rotates by n_pairs % n_cta per simulation, so that with a CTA
                              // count that does not divide the pair count every CTA gets the extra pass equally often
};
#ifdef HMZ_PERSIST_STATS  // tooling build (tools/build_variant.py): role statistics of the persistent kernel
constexpr bool kPersistStats = true;
#else
constexpr bool kPersistStats = false;
#endif
// Back-off between two polls of a hand-off word (ns; 0 = poll back to back).  Tuning switch.
#ifdef HMZ_PERSIST_SLEEP_NS
#define HMZ_PERSIST_SLEEP_NS_SET 1  // (hmz_build_flags reports a non-default value)
#else
#define HMZ_PERSIST_SLEEP_NS 64
#endif
__device__ __forceinline__ void persist_backoff() {
  if (HMZ_PERSIST_SLEEP_NS > 0) __nanosleep(HMZ_PERSIST_SLEEP_NS);
}
constexpr int kSlicesPerPair = 16;       // warps (16 searches each) per 256-search tile pair
__device__ __forceinline__ uint32_t ld_relaxed_u32(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned long long ld_relaxed_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
// Leaf parents / actions: written by the PREVIOUS kernel (stand-alone launches: plain loads) or by other CTAs of the
// same kernel (persistent schedule: L1-bypassing relaxed loads, never the read-only path).
template <bool kPersist>
__device__ __forceinline__ uint32_t ld_leaf_u16(const uint16_t* p) {
  if (!kPersist) return *p;
  uint32_t v;
  asm volatile("ld.relaxed.gpu.global.u16 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
template <bool kPersist>
__device__ __forceinline__ uint32_t ld_leaf_u8(const uint8_t* p) {
  if (!kPersist) return *p;
  uint32_t v;
  asm volatile("ld.relaxed.gpu.global.u8 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void fence_acquire_gpu() { asm volatile("fence.acquire.gpu;" ::: "memory"); }
__device__ __forceinline__ void red_release_add(uint32_t* p, uint32_t v) {
  asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void st_release_u64(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
// Every thread that is about to read what the tree warps wrote for (pair, sim) — leaf parents / actions — calls this:
// polls the pair's counter (relaxed, L2) until all 16 slices of that simulation's selection are done, then acquires.
__device__ __forceinline__ void persist_wait_tree(const PersistCtl& pc, int pair, int sim) {
  const uint32_t need = (uint32_t)kSlicesPerPair * (uint32_t)(sim + 1);
  const uint32_t* ctr = pc.tree_done + (size_t)pair * 8;
  WaitGuard guard;
  while (ld_relaxed_u32(ctr) < need) {
    persist_backoff();
    guard.poll();
#ifdef HMZ_WATCHDOG_SOFT
    if (guard.expired) {
      if ((threadIdx.x & 127) == 0) printf("MLP cta %d thread %d: pair %d sim %d waits tree_done >= %u, sees %u\n", (int)blockIdx.x, (int)threadIdx.x, pair, sim, need, ld_relaxed_u32(ctr));
      break;
    }
#endif
  }
  fence_acquire_gpu();
}
// One thread, after every output of (pair, sim) is in global memory and ordered before it at CTA scope: hands the pair
// to the tree warps as work item (pair, sim + 1).
__device__ __forceinline__ void persist_push_item(const PersistCtl& pc, int n_pairs, int pair, int sim_next) {
  if (pc.mlp_done != nullptr) {  // server schedule: the pair's flag is the hand-off
    asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(pc.mlp_done + (size_t)pair * 8), "r"((uint32_t)sim_next) : "memory");
    if (pc.group_done != nullptr) red_release_add(pc.group_done + (size_t)(pair / pc.pairs_per_group) * 8, 1u);
    return;
  }
  const uint32_t pos = atomicAdd(pc.q_tail, 1u);
  const unsigned long long item = (unsigned long long)n_pairs + pos;
  st_release_u64(pc.queue + (pos & pc.q_mask), ((item + 1ull) << 32) | (unsigned long long)((uint32_t)pair | ((uint32_t)sim_next << 16)));
}

// kInitial = false: recurrent_inference — networks dynamics (g), reward, policy, value; input = gathered latents.
// kInitial = true : initial_inference  — networks representation (h), policy, value; input = one-hot of env words.
// kPersist = true : MLP role of the persistent search kernel: CTA `cta` of `n_cta` owns tile pairs cta, cta + n_cta, ...
//                   and runs them once per simulation, in that order; a pass (pair, sim) starts when the tree warps have
//                   finished the pair's selection of simulation sim and ends by handing the pair back (persist_push_item).
// The network index `net` keeps the recurrent numbering (0 = g / h, 1 = reward, 2 = policy, 3 = value);
// the root inference simply skips net 1.
template <bool kInitial, bool kPersist>
__device__ __forceinline__ void net_tc_body(const TcArgs& a, const PersistCtl& pc, uint8_t* smem_raw, int cta_raw, int n_cta_raw) {
  // head split (TcArgs::head_split): `cta` / `n_cta` below count tile-pair owners; role -1 = all networks
  const int split = (!kInitial && !kPersist && a.head_split == 3) ? 3 : 1;
  const int role = split == 3 ? cta_raw % 3 : -1;
  const int cta = cta_raw / split, n_cta = n_cta_raw / split;
  auto runs = [&](int net) { return net == 0 || split == 1 || net == role + 1; };
  const uint8_t* __restrict__ wsec = a.wsec;
  const void* __restrict__ lat_in = a.lat_in;
  const int64_t in_rows_per_item = a.in_rows_per_item;
  const uint16_t* __restrict__ in_row = a.in_row;
  const uint8_t* __restrict__ actions = a.actions;
  const uint32_t* __restrict__ words = a.words;
  const int n_disks = a.n_disks;
  void* lat_out = a.lat_out;
  const int64_t out_rows_per_item = a.out_rows_per_item;
  const int latent_dtype = a.latent_dtype;
  float* __restrict__ r_out = a.r_out;
  float* __restrict__ p_out = a.p_out;
  float* __restrict__ v_out = a.v_out;
  const int64_t n = a.n;
  const int n_pairs = a.n_pairs;
  const int timeline = a.timeline;  // (persistent passes: only the tooling bits 0 and 8+ are set)
  // passes of this CTA: its tile pairs, once (stand-alone) or once per simulation (persistent)
  // (pair, sim) sequence of this CTA: in simulation s it owns the pairs first_pair(s), first_pair(s) + n_cta, ...
  const int rot = (kPersist && pc.rotate) ? n_pairs % n_cta : 0;
  auto first_pair = [&](int sim) {
    int f = cta - (int)(((long long)sim * rot) % n_cta);
    return f < 0 ? f + n_cta : f;
  };
  int n_pass = 0;
  if (kPersist && rot != 0) {
    for (int sm = 0; sm < pc.n_sims; ++sm) {
      const int f = first_pair(sm);
      if (f < n_pairs) n_pass += (n_pairs - f - 1) / n_cta + 1;
    }
  } else {
    const int own = cta < n_pairs ? (n_pairs - cta + n_cta - 1) / n_cta : 0;
    n_pass = kPersist ? own * pc.n_sims : own;
  }
  struct PassIter {
    int pair, sim;
  };
  auto next_item = [&](PassIter& it) {
    it.pair += n_cta;
    while (it.pair >= n_pairs && it.sim + 1 < (kPersist ? pc.n_sims : 1)) {
      ++it.sim;
      it.pair = first_pair(it.sim);
    }
  };
  Smem& s = *reinterpret_cast<Smem*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int tid = threadIdx.x, warp = tid >> 5;
// (the clock is read through an asm with a memory clobber so that it cannot be scheduled above a barrier)
#define TL4_CTA(slot)                                                        \
  do {                                                                       \
    if ((timeline & 1) && cta == 0 && tid == 0) {                     \
      unsigned long long now_;                                               \
      asm volatile("mov.u64 %0, %%clock64;" : "=l"(now_)::"memory");         \
      g_timeline[slot] = now_;                                               \
    }                                                                        \
  } while (0)
  TL4_CTA(60);
  if (!kPersist && tid == 0) gantt_mark(a.gantt, 0);

  // barrier initialisation is spread over one lane of each of warps 1-3 while warp 0 allocates TMEM
  if (tid == 32) {
    for (int k = 0; k < 2; ++k)
      for (int j = 0; j < 2; ++j) {
        mbar_init(&s.bar_wfull[k][j], 1);
        mbar_init(&s.bar_wfree[k][j], 2);  // one commit per tile's MMA warp
      }
    mbar_init(&s.bar_end, 2);
    mbar_init(&s.bar_pass, 2 * kHidThreadsPerTile + 128);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (tid == 64 || tid == 96) {
    const int t = (tid >> 5) - 2;
    mbar_init(&s.bar_g[t], kHidThreadsPerTile + 128);
    mbar_init(&s.bar_d[t], 1);
    mbar_init(&s.bar_a[t], kHidThreadsPerTile);
    mbar_init(&s.bar_o[t], 1);
    mbar_init(&s.bar_s[t], 1);
    mbar_init(&s.bar_raw[t], kHidThreadsPerTile);
    mbar_init(&s.bar_hn[t], kHidThreadsPerTile);
    mbar_init(&s.bar_fin[t], 128);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {  // TMEM: all 512 columns (one CTA per SM)
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&s.tmem_base)), "r"(512u)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = s.tmem_base;
  TL4_CTA(61);
  // Programmatic dependent launch: barrier init, TMEM allocation and (loader warp) the first weight
  // blocks do not depend on the preceding tree kernel; everything that reads its outputs does.
  // The dependents (the next tree kernel) are signalled only AFTER this kernel's own wait: that kernel reads
  // what the previous tree kernel wrote before it waits for this one, so it must not start before the
  // previous tree kernel has completed.  (The loader warp waits after its first four weight blocks.)
  const bool late_signal = !kPersist && (timeline & 2) != 0;  // HMZ_PDL bit 2
  const int signal_net = kPersist ? 8 : ((timeline >> 2) & 7) - 1;  // HMZ_PDL_NET_AT: -1 = here (8: never)
  if (!kPersist) {
    if (!late_signal && signal_net < 0) pdl_launch_dependents();
    if (warp != kLoaderWarp && (late_signal || (warp != kMmaWarp && warp != kMmaWarp1))) {
      pdl_wait();
      if (late_signal && signal_net < 0) pdl_launch_dependents();
    }
  }
  TL4_CTA(62);

  if (warp == kLoaderWarp) {
    // ================================= loader warp =================================
    // Block i = 2 * network + layer goes to slot (network & 1) of its kind, so that the second-layer slot 1 only ever
    // holds the reward / policy blocks; cnt = loads issued into a slot so far (a reload waits for the previous use's MMAs).
    uint32_t cnt[2][2] = {{0u, 0u}, {0u, 0u}};
    int issued = 0;
    PassIter load_it{first_pair(0), 0};  // the pair of the pass whose blocks are loaded (the MMA warps may still run the one before)
    for (int pass = 0; pass < n_pass; ++pass, next_item(load_it)) {
      const uint8_t* __restrict__ wpass = (!kPersist && a.block_set != nullptr) ? wsec + (int64_t)a.block_set[load_it.pair] * a.weight_stride : wsec;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        if (kInitial && (i >> 1) == 1) continue;  // no reward head at the root
        if (!runs(i >> 1)) continue;
        if (late_signal && pass == 0 && issued == (split == 1 ? 4 : 2)) {  // the first blocks are in flight: now order after the preceding kernel
          pdl_wait();
          if (signal_net < 0) pdl_launch_dependents();
        }
        ++issued;
        const int kind = i & 1, slot = (i >> 1) & 1;
        const uint32_t u = cnt[kind][slot];
        if (u >= 1u) mbar_wait(&s.bar_wfree[kind][slot], (u - 1u) & 1u);
        const uint32_t off = (kInitial && i < 2) ? (i == 0 ? kWh1 : kWh2) : c_block_off[i];  // representation_net at the root
        uint8_t* dst = kind ? (slot ? s.ws1 : s.ws0) : s.wf[slot];
        if (elect_one()) tma_load(dst, wpass + off, c_block_bytes[i], &s.bar_wfull[kind][slot]);
        __syncwarp();
        cnt[kind][slot] = u + 1u;
      }
    }
  } else if (warp == kMmaWarp || warp == kMmaWarp1) {
    // ================================= MMA-issuing warps =================================
    // One warp per tile; an elected lane issues the tile's tcgen05.mma instructions  L1 L2  per network.  Issuing is
    // blocking (~50 clk per small second-layer instruction, tools/microbench/mma.cu), so with one warp per tile a
    // tile's waits and issue slots never sit behind the other tile's; the tensor core interleaves the two streams.
    const int t = warp == kMmaWarp ? 0 : 1;
    const uint32_t id256 = umma_idesc(256);
    const uint32_t T = tmem + kColsPerTile * t;
    const uint32_t ax = smem_u32(s.t[t].ax);
    uint32_t use0 = 0, use1 = 0, ph_g = 0, ph_a = 0, ph_raw = 0, ph_hn = 0, ph_fin = 0;  // use0 / use1: networks done on weight slot 0 / 1
    bool first = true;
    for (int pass = 0; pass < n_pass; ++pass) {
#pragma unroll 1
      for (int net = 0; net < 4; ++net) {  // dynamics / representation, reward, value, policy
        if (kInitial && net == 1) continue;
        if (!runs(net)) continue;
        if (t == 0 && net == signal_net && pass == n_pass - 1) pdl_launch_dependents();
        // ---- first layer: H[0:256) = [A | AX] x W1'^T
        {
          const uint32_t slot = (uint32_t)net & 1u, use = slot ? use1 : use0;  // both layers of a network use slot (net & 1)
          if (elect_one()) TL4(16 + net * 2 + t);
          mbar_wait(&s.bar_wfull[0][slot], use & 1u);
          const uint32_t wf = smem_u32(s.wf[slot]);
          const uint32_t a_in = net <= 1 ? smem_u32(s.t[t].a0) : smem_u32(s.t[t].ahn);
          if (net == 0) mbar_wait(&s.bar_g[t], ph_g);
          if (net == 1) mbar_wait(&s.bar_raw[t], ph_raw);  // raw latent tile written, O copied out
          if (net == 2 || (net == 3 && split == 3)) mbar_wait(&s.bar_hn[t], ph_hn);  // normalised latent tile written
          // O (inside H) must have been copied out: by the output warps after a head, by the latent epilogue
          // (bar_raw / bar_hn above) after the first network.  (Head split: one head and one pass per CTA — nothing to wait for.)
          if (split == 1 && (net == 3 || (net == 2 && !kInitial) || (net == 0 && !first))) {
            mbar_wait(&s.bar_fin[t], ph_fin);
            ph_fin ^= 1;
          }
          if (elect_one()) TL4(net * 4 + t);
          tc_fence_after();
          if (elect_one()) {
            // one N = 256 instruction per k-step: A is fetched from shared memory once for both column
            // halves (two N = 128 instructions read it twice and saturate the shared-memory port)
            const uint64_t a_base = desc_sw128(a_in), b_base = desc_sw128(wf);
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) umma(T, a_base + (uint64_t)(kk * 2), b_base + (uint64_t)(kk * 2), id256, kk ? 1u : 0u);
            umma(T, desc_plain(ax), desc_plain(wf + 256 * 128), id256, 1u);
            umma_commit(&s.bar_d[t]);
            umma_commit(&s.bar_wfree[0][slot]);
          }
          __syncwarp();
          if (net == 0) ph_g ^= 1;
          if (net == 1) ph_raw ^= 1;
          if (net == 2) ph_hn ^= 1;
        }
        // ---- second layer: O = [A1 | AX] x W2'^T, A1 from TMEM
        {
          const uint32_t n2 = net == 0 ? 64u : (net == 3 ? 16u : 48u);
          const uint32_t id2 = umma_idesc(n2);
          const uint32_t slot = (uint32_t)net & 1u, use = slot ? use1 : use0;
          mbar_wait(&s.bar_wfull[1][slot], use & 1u);
          const uint32_t ws = smem_u32(slot ? s.ws1 : s.ws0);
          mbar_wait(&s.bar_a[t], ph_a);
          if (elect_one()) TL4(net * 4 + 2 + t);
          tc_fence_after();
          if (elect_one()) {
            umma(T + kColO, desc_plain(ax), desc_plain(ws + n2 * 128 * 4), id2, 0u);  // bias step clears O
            const uint64_t b_base = desc_sw128(ws);
#pragma unroll
            for (int j = 0; j < 16; ++j)
              umma_ts(T + kColO, T + (j >> 3) * kColH1 + (j & 7) * 8,
                      b_base + (uint64_t)(((j >> 2) * n2 * 128 + (j & 3) * 32) >> 4), id2, 1u);
            umma_commit(net == 0 ? &s.bar_o[t] : &s.bar_s[t]);
            umma_commit(&s.bar_wfree[1][slot]);
          }
          __syncwarp();
          ph_a ^= 1;
          if (slot) ++use1; else ++use0;
        }
      }
      first = false;
    }
    if (elect_one()) umma_commit(&s.bar_end);
    __syncwarp();
    mbar_wait(&s.bar_end, 0);
  } else if (warp > kMmaWarp1) {
    // spare warp (CTAs launched with 24 warps: the persistent kernel): nothing to do
  } else if (warp < kSmallWarp0) {
    // ============================== hidden-epilogue warps ==============================
    const int t = warp >> 3, ltid = tid & 255;
    const int row = ltid & 127, half = ltid >> 7, quarter = warp & 3;
    Tile& tile = s.t[t];
    const uint32_t lane_bits = (uint32_t)(quarter * 32) << 16;
    const uint32_t T = tmem + kColsPerTile * t + lane_bits;
    uint32_t ph_d = 0, ph_o = 0;
    bool copy_pending = false;
    PassIter item_it{first_pair(0), 0};
    for (int pass = 0; pass < n_pass; ++pass, next_item(item_it)) {
      const int pair = item_it.pair, sim = item_it.sim;
      const int64_t out_row = kPersist ? (int64_t)sim + 1 : a.out_row;
      const int64_t row0 = ((int64_t)pair * 2 + t) * kM;
      const int64_t item = row0 + row;
      if (ltid == 0 && t == 0) TL4(64);
      if (kPersist) {  // the gather reads what the pair's selection wrote
        const bool st = kPersistStats && pc.stats != nullptr && ltid == 0 && t == 0;
        const long long c0 = st ? clock64() : 0;
        persist_wait_tree(pc, pair, sim);
        if (st) {
          atomicAdd(pc.stats + 4, (unsigned long long)(clock64() - c0));
          atomicAdd(pc.stats + 6, 1ull);
        }
      }
      {  // parent latents -> swizzled A0 tile; 8 consecutive lanes fetch the 8 16-byte chunks of one row
        const int chunk = ltid & 7;
        uint4 gathered[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int grow = (ltid >> 3) + 32 * i;
          const int64_t it = (row0 + grow) < n ? (row0 + grow) : n - 1;
          if (kInitial) {  // utils.oneHot_encoding (utils.py:9-25) of the env word: columns 8 chunk .. 8 chunk + 7
            const uint32_t w = words[it];
            uint32_t v[4] = {0u, 0u, 0u, 0u};
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const int col = chunk * 8 + j, d = col / 3;
              if (col < 3 * n_disks && ((w >> (2 * d)) & 3u) == (uint32_t)(col - 3 * d)) v[j >> 1] |= 0x3F80u << ((j & 1) * 16);
            }
            gathered[i] = make_uint4(v[0], v[1], v[2], v[3]);
            continue;
          }
          const int64_t irow = it * in_rows_per_item + (in_row ? (int64_t)ld_leaf_u16<kPersist>(in_row + it) : 0);
          if (latent_dtype == HMZ_LATENT_F32) {
            const float4* src = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(lat_in) + irow * kLatent + chunk * 8);
            const float4 t0 = __ldcs(src), t1 = __ldcs(src + 1);
            gathered[i] = make_uint4(pack_bf16(t0.x, t0.y), pack_bf16(t0.z, t0.w), pack_bf16(t1.x, t1.y), pack_bf16(t1.z, t1.w));
          } else {
            gathered[i] = __ldcs(reinterpret_cast<const uint4*>(reinterpret_cast<const uint16_t*>(lat_in) + irow * kLatent + chunk * 8));
          }
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) *reinterpret_cast<uint4*>(tile.a0 + sw128((ltid >> 3) + 32 * i, chunk)) = gathered[i];
        fence_proxy_async();
        mbar_arrive(&s.bar_g[t]);
        if (ltid == 0) TL4(80 + t * 8);
      }
#pragma unroll 1
      for (int layer = 0; layer < 4; ++layer) {
        if (kInitial && layer == 1) continue;
        if (!runs(layer)) continue;
        mbar_wait(&s.bar_d[t], ph_d);
        ph_d ^= 1;
        tc_fence_after();
        hidden_epilogue_tmem(T + half * kColH1);
        tc_fence_before();
        mbar_arrive(&s.bar_a[t]);
        if (ltid == 0) TL4(81 + t * 8 + layer);
        if (layer == 0) {
          // ---- new latent: normalize_h_state (networks.py:191-196) and its copies; thread (row, half)
          // owns latent columns [32*half, 32*half + 32)
          mbar_wait(&s.bar_o[t], ph_o);
          ph_o ^= 1;
          tc_fence_after();
          if (ltid == 0) TL4(44 + t * 8);
          float raw[32];
          tmem_ld32(T + kColO + half * 32, raw);
          // the raw latent feeds the reward head: publish it first so that head's MMA overlaps the rest
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            uint32_t pr[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) pr[j] = pack_bf16(raw[c * 8 + 2 * j], raw[c * 8 + 2 * j + 1]);
            *reinterpret_cast<uint4*>(tile.a0 + sw128(row, half * 4 + c)) = make_uint4(pr[0], pr[1], pr[2], pr[3]);
          }
          fence_proxy_async();
          tc_fence_before();
          mbar_arrive(&s.bar_raw[t]);
          if (ltid == 0) TL4(86 + t * 8);
          float mn4[4], mx4[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) mn4[i] = mx4[i] = raw[i];
#pragma unroll
          for (int i = 4; i < 32; ++i) {
            mn4[i & 3] = fminf(mn4[i & 3], raw[i]);
            mx4[i & 3] = fmaxf(mx4[i & 3], raw[i]);
          }
          s.row_minmax[t][half][row] = make_float2(fminf(fminf(mn4[0], mn4[1]), fminf(mn4[2], mn4[3])),
                                                   fmaxf(fmaxf(mx4[0], mx4[1]), fmaxf(mx4[2], mx4[3])));
          asm volatile("bar.sync %0, 64;" ::"r"(1 + t * 4 + quarter) : "memory");
          if (ltid == 0) TL4(40 + t * 8);
          const float2 m0 = s.row_minmax[t][0][row], m1 = s.row_minmax[t][1][row];
          const float mn = fminf(m0.x, m1.x), mx = fmaxf(m0.y, m1.y);
          const float inv = 1.0f / ((mx - mn) + 1e-8f);
          const int64_t orow = item * out_rows_per_item + out_row;
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            float hn[8];
            uint32_t ph[4];
#pragma unroll
            for (int j = 0; j < 8; ++j) hn[j] = (raw[c * 8 + j] - mn) * inv;
#pragma unroll
            for (int j = 0; j < 4; ++j) ph[j] = pack_bf16(hn[2 * j], hn[2 * j + 1]);
            *reinterpret_cast<uint4*>(tile.ahn + sw128(row, half * 4 + c)) = make_uint4(ph[0], ph[1], ph[2], ph[3]);
            if (latent_dtype == HMZ_LATENT_F32 && item < n && role <= 0) {  // parity-mode stores keep the per-row form
              float4* dst = reinterpret_cast<float4*>(reinterpret_cast<float*>(lat_out) + orow * kLatent + half * 32 + c * 8);
              __stcs(dst, make_float4(hn[0], hn[1], hn[2], hn[3]));
              __stcs(dst + 1, make_float4(hn[4], hn[5], hn[6], hn[7]));
            }
          }
          if (ltid == 0) TL4(41 + t * 8);
          fence_proxy_async();
          mbar_arrive(&s.bar_hn[t]);
          if (ltid == 0) TL4(42 + t * 8);
          copy_pending = true;  // the rows leave for HBM after the NEXT hidden drain (see below)
        } else if (copy_pending) {
          // ---- deferred copy-out of the new latent rows (bf16): issued after the first head's hidden drain, while this
          // tile's second-layer MMA runs, so that it no longer delays that drain (it did, by ~1,400 clk per pass).
          // The normalised tile is only read by the remaining heads' first layers, never rewritten within the pass.
          copy_pending = false;
          if (latent_dtype != HMZ_LATENT_F32) {
            // 8 consecutive lanes write one 128-byte row: the two warps of a lane quarter copy out 16 rows each,
            // once both have written their column halves of the tile
            asm volatile("bar.sync %0, 64;" ::"r"(1 + t * 4 + quarter) : "memory");
            const int lane = tid & 31, chunk = lane & 7;
            if (ltid == 0) TL4(43 + t * 8);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const int r2 = quarter * 32 + half * 16 + i * 4 + (lane >> 3);
              const int64_t it2 = row0 + r2;
              const uint4 val = *reinterpret_cast<const uint4*>(tile.ahn + sw128(r2, chunk));
              if (it2 < n && role <= 0)  // (head split: the reward CTA stores the rows)
                __stcs(reinterpret_cast<uint4*>(reinterpret_cast<uint16_t*>(lat_out) + (it2 * out_rows_per_item + out_row) * kLatent + chunk * 8), val);
            }
          }
          if (ltid == 0) TL4(85 + t * 8);
          if (kPersist) mbar_arrive(&s.bar_pass);  // this thread's latent stores of the pass are issued
        }
      }
    }
  } else {
    // ============================== output warps (both tiles) ==============================
    const int row = tid - kSmallWarp0 * 32;
    const uint32_t lane_bits = (uint32_t)((warp & 3) * 32) << 16;
    uint32_t ph_s = 0;
    uint32_t ph_pass = 0;
    unsigned long long pass_t0 = 0;
    PassIter item_it{first_pair(0), 0};
    for (int pass = 0; pass < n_pass; ++pass, next_item(item_it)) {
      const int pair = item_it.pair, sim = item_it.sim;
      if (kPersist) persist_wait_tree(pc, pair, sim);  // the action slice reads what the pair's selection wrote
#pragma unroll
      for (int t = 0; t < 2; ++t) {  // the extra A slice of this row: one-hot(action) at k = 0..5, the constant 1 at k = 6
        const int64_t item = ((int64_t)pair * 2 + t) * kM + row;
        uint32_t w[4] = {0u, 0u, 0u, 0x3F80u};  // k = 6 -> 1.0 (bf16 0x3F80), k = 7 -> 0
        if (!kInitial) {
          int act = (int)ld_leaf_u8<kPersist>(actions + (item < n ? item : n - 1));
          act = act < kActions ? act : kActions - 1;
          w[act >> 1] |= 0x3F80u << ((act & 1) * 16);
        }
        *reinterpret_cast<uint4*>(s.t[t].ax + plain_off(row, 0)) = make_uint4(w[0], w[1], w[2], w[3]);
        *reinterpret_cast<uint4*>(s.t[t].ax + plain_off(row, 1)) = make_uint4(0u, 0u, 0u, 0u);
        fence_proxy_async();
        mbar_arrive(&s.bar_g[t]);
      }
#pragma unroll 1
      for (int head = 0; head < 3; ++head) {  // reward, value, policy
        if (kInitial && head == 0) continue;
        if (!runs(head + 1)) continue;
#pragma unroll 1
        for (int t = 0; t < 2; ++t) {
          const int64_t item = ((int64_t)pair * 2 + t) * kM + row;
          const uint32_t O = tmem + kColsPerTile * t + kColO + lane_bits;
          mbar_wait(&s.bar_s[t], ph_s);
          tc_fence_after();
          if (head == 2) {  // F.softmax(pi_logits) (networks.py:109)
            float lg[16];
            tmem_ld16(O, lg);
            tc_fence_before();
            mbar_arrive(&s.bar_fin[t]);
            float mx = lg[0], den = 0.f;
#pragma unroll
            for (int a = 1; a < kActions; ++a) mx = fmaxf(mx, lg[a]);
#pragma unroll
            for (int a = 0; a < kActions; ++a) {
              lg[a] = exp2f((lg[a] - mx) * 1.4426950408889634f);
              den += lg[a];
            }
            const float inv = 1.0f / den;
            if (item < n) {
#pragma unroll
              for (int a = 0; a < kActions; ++a) p_out[item * kActions + a] = lg[a] * inv;
            }
          } else {  // softmax expectation over the 33 support logits + signed parabolic (networks.py:152-189)
            float a[32], b[16];
            tmem_ld32(O, a);
            tmem_ld16(O + 32, b);
            tc_fence_before();
            mbar_arrive(&s.bar_fin[t]);
            float m4[4] = {a[0], a[1], a[2], a[3]};
#pragma unroll
            for (int i = 4; i < 32; ++i) m4[i & 3] = fmaxf(m4[i & 3], a[i]);
            const float mx = fmaxf(fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3])), b[0]);
            const float ms = mx * 1.4426950408889634f;
            float den4[4] = {0.f, 0.f, 0.f, 0.f}, num4[4] = {0.f, 0.f, 0.f, 0.f};  // four independent chains
#pragma unroll
            for (int i = 0; i < 32; ++i) {
              const float e = exp2f(fmaf(a[i], 1.4426950408889634f, -ms));
              den4[i & 3] += e;
              num4[i & 3] = fmaf(e, (float)(i - 16), num4[i & 3]);
            }
            const float e = exp2f(fmaf(b[0], 1.4426950408889634f, -ms));
            const float den = ((den4[0] + den4[1]) + (den4[2] + den4[3])) + e;
            const float num = fmaf(e, 16.f, (num4[0] + num4[1]) + (num4[2] + num4[3]));
            const float x = signed_parabolic(__fdividef(num, den));
            if (item < n) (head == 0 ? r_out : v_out)[item] = x;
          }
          if (row == 0) TL4(70 + head * 2 + t);
        }
        ph_s ^= 1;
      }
      if (kPersist) {
        // every r / p / v store of the pass is issued; thread 0 of the output warps waits until the 512 latent-writing
        // threads and the 128 output threads have arrived (release / acquire at CTA scope), then publishes the pair with
        // a GPU-scope release: the tree warps that take it see every output of the pass.
        mbar_arrive(&s.bar_pass);
        if (row == 0) {
          mbar_wait(&s.bar_pass, ph_pass);
          persist_push_item(pc, n_pairs, pair, sim + 1);
          TL4(66);
          if (kPersistStats && pc.stats != nullptr) {
            const unsigned long long now = (unsigned long long)clock64();
            if (pass == 0) pass_t0 = now;
            if (pass == n_pass - 1) atomicAdd(pc.stats + 5, now - pass_t0);  // first push -> last push of this CTA
          }
        }
        ph_pass ^= 1;
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  TL4_CTA(63);
  if (!kPersist && tid == 0) gantt_mark(a.gantt, 1);
  if (warp == 0) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512u) : "memory");
  }
}
#undef TL4_CTA

#undef TL4
}  // namespace v4
}  // namespace tc
}  // namespace hmz
