// Shared host/device helpers for libhmz.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>

#include "hmz.h"

namespace hmz {

constexpr int kSmFallback = 148;  // B200: 148 SMs (2 dies x 74)

// ---- error plumbing (never throw across the C ABI) -------------------------------------
char* error_buffer();                       // thread-local, 512 bytes
int fail(int code, const char* fmt, ...);   // formats into error_buffer(), returns code
extern std::atomic<long long> g_launches;   // kernels launched by this process

inline int check_launch(const char* what) {
  g_launches.fetch_add(1, std::memory_order_relaxed);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(HMZ_ERR_CUDA, "%s: %s", what, cudaGetErrorString(e));
  return HMZ_OK;
}

// RAII CUDA-event bracket around the launches of one extern "C" entry point (hmz_prof_*).
extern std::atomic<int> g_prof_on;
void prof_push(int cls, cudaStream_t stream, bool start);
struct ProfScope {
  int cls;
  cudaStream_t stream;
  bool on;
  ProfScope(int c, void* s) : cls(c), stream((cudaStream_t)s), on(g_prof_on.load(std::memory_order_relaxed) != 0) {
    if (on) prof_push(cls, stream, true);
  }
  ~ProfScope() {
    if (on) prof_push(cls, stream, false);
  }
};

// Programmatic dependent launch (PDL): the kernel may start while its stream predecessor drains; it
// must execute pdl_wait() before touching anything the predecessor produced (or still reads).
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// Launches `kernel` as a programmatic dependent of its stream predecessor.  The network kernels and the tree
// kernel launch this way; each signals its own dependents early (see net_tc_body and tree_phase).
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                              Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// Tooling (hmz_debug_gantt): when recording is on, the next launch of a hot-loop kernel by this host thread gets a slot of
// two device words — the globaltimer of its first block's start and (complemented, so that both are atomicMin) of its
// last block's end.  gantt_next() hands out the slot and remembers (kind, tag); nullptr when recording is off.
unsigned long long* gantt_next(int kind, int tag);
__device__ __forceinline__ void gantt_mark(unsigned long long* slot, int which) {
  if (slot != nullptr) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    atomicMin(slot + which, which ? ~t : t);
  }
}
// (kind, tag) of the launch being enqueued by this host thread: set by hmz_search_run around each launch
void gantt_set_context(int group, int sim);
int gantt_context_tag();

int sm_count();  // cached cudaDevAttrMultiProcessorCount of the current device (148 on B200)

// Grid for a grid-stride kernel: a whole number of waves of `ctas_per_sm` CTAs on every SM,
// never more CTAs than there is work for.
inline unsigned grid_for(int64_t work_items, int items_per_cta, int ctas_per_sm) {
  int64_t need = (work_items + items_per_cta - 1) / items_per_cta;
  int64_t wave = (int64_t)sm_count() * ctas_per_sm;
  if (need <= wave) return (unsigned)(need < 1 ? 1 : need);
  int64_t waves = (need + wave - 1) / wave;
  if (waves > 8) waves = 8;  // beyond 8 waves the grid-stride loop takes over
  return (unsigned)(waves * wave);
}

// ---- Philox4x32-10 (counter-based RNG; Salmon et al. 2011) ------------------------------
struct Philox4 {
  uint32_t x, y, z, w;
};

__host__ __device__ __forceinline__ uint32_t mulhi32(uint32_t a, uint32_t b) {
#ifdef __CUDA_ARCH__
  return __umulhi(a, b);
#else
  return (uint32_t)(((uint64_t)a * b) >> 32);
#endif
}

__host__ __device__ __forceinline__ Philox4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                          uint32_t k0, uint32_t k1) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0 = mulhi32(M0, c0), lo0 = M0 * c0;
    uint32_t hi1 = mulhi32(M1, c2), lo1 = M1 * c2;
    uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += W0; k1 += W1;
  }
  return Philox4{c0, c1, c2, c3};
}

}  // namespace hmz
