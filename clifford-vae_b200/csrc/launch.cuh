// Host-side launch plumbing shared by the api_*.cu translation units.
#pragma once
#include <cstdio>
#include <atomic>
#include <type_traits>
#include "common.cuh"
#include "rng.cuh"

namespace cvb {

void set_last_error(const char* fmt, ...);
// Device twiddle table for the current device (nullptr + error set if cvb_init() was not called).
const cplx* device_twiddles();
int sm_count();
// A zero-initialised (next-row, finished-groups) counter pair for one dynamically scheduled launch; a ring of 64
// pairs lets launches on different streams overlap (each kernel re-arms its pair when its last group finishes).
int* next_sched_slot();
extern std::atomic<long long> g_launch_count;

#define CVB_REQUIRE(cond, code, ...)          \
  do {                                        \
    if (!(cond)) {                            \
      ::cvb::set_last_error(__VA_ARGS__);     \
      return code;                            \
    }                                         \
  } while (0)

#define CVB_CUDA(call)                                                                   \
  do {                                                                                   \
    cudaError_t e_ = (call);                                                             \
    if (e_ != cudaSuccess) {                                                             \
      ::cvb::set_last_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
      return ::cvb::kCudaError;                                                          \
    }                                                                                    \
  } while (0)

inline int check_launch(const char* what) {
  g_launch_count.fetch_add(1, std::memory_order_relaxed);
  cudaError_t e = cudaPeekAtLastError();
  if (e != cudaSuccess) {
    cudaGetLastError();
    set_last_error("launch of %s failed: %s", what, cudaGetErrorString(e));
    return kCudaError;
  }
  return kOk;
}

// Persistent grid: min(work CTAs, SMs x resident CTAs per SM).  Opts in to > 48 KB dynamic smem.
// The > 48 KB opt-in is tracked per (device, kernel) and only ever raised; the occupancy answer is cached per
// (device, kernel, threads, smem) -- kernels with a run-time shared-memory size are launched with several sizes.
int cached_ctas_per_sm(const void* kernel, int threads, size_t smem, bool* found);
void store_ctas_per_sm(const void* kernel, int threads, size_t smem, int per_sm);
int ensure_smem_optin(const void* kernel, size_t smem);

template <typename Kernel>
inline int persistent_grid(Kernel kernel, int threads, size_t smem, long long work_ctas, int* grid_out) {
  bool found = false;
  int per_sm = cached_ctas_per_sm(reinterpret_cast<const void*>(kernel), threads, smem, &found);
  if (!found) {
    if (int rc = ensure_smem_optin(reinterpret_cast<const void*>(kernel), smem)) return rc;
    CVB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, smem));
    store_ctas_per_sm(reinterpret_cast<const void*>(kernel), threads, smem, per_sm);
  }
  if (per_sm < 1) {
    set_last_error("kernel does not fit on an SM (threads=%d smem=%zu)", threads, smem);
    return kUnsupported;
  }
  long long g = (long long)sm_count() * per_sm;
  if (g > work_ctas) g = work_ctas;
  if (g < 1) g = 1;
  *grid_out = (int)g;
  return kOk;
}

// device launch counter registered for the current device (nullptr when none), see cvb_set_rng_device_counter
const unsigned long long* rng_device_counter();
// arrival word of the self-bumping mode for the current device (nullptr unless cvb_set_rng_device_counter_autobump is active)
unsigned int* rng_arrive_word();

inline PhiloxKey make_key(unsigned long long seed, unsigned long long offset, uint32_t stream_id) {
  PhiloxKey k;
  k.dev_counter = rng_device_counter();
  k.arrive = k.dev_counter ? rng_arrive_word() : nullptr;
  k.k0 = (uint32_t)seed;
  k.k1 = (uint32_t)(seed >> 32);
  k.offset = (uint32_t)offset ^ (uint32_t)((offset >> 32) * 0x9E3779B9u);
  k.stream = stream_id;
  philox_fill_round_keys(k);
  return k;
}

// Persistent launch: persistent_grid -> launch -> check_launch.  `args` are the kernel's arguments.
template <typename Kernel, typename... Args>
inline int launch_persistent(Kernel kern, const char* what, int threads, size_t smem, long long work, cudaStream_t st,
                             const Args&... args) {
  int grid = 0;
  if (int rc = persistent_grid(kern, threads, smem, work, &grid)) return rc;
  kern<<<grid, threads, smem, st>>>(args...);
  return check_launch(what);
}

// The same with programmatic dependent launch (sm_90+): the kernel is allowed to become resident while its predecessor
// on the stream drains; it blocks at pdl_wait_and_release() (griddepcontrol.wait) -- its first statement, before any
// global access to caller data -- until the predecessor has completed and flushed.  That removes the launch / scheduling
// gap between the back-to-back kernels of a step (sampler -> bind -> sampler ...).  Only for kernels that begin with
// pdl_wait_and_release(): one without the wait would read its inputs before the predecessor has written them.
// `sched` (or null): the schedule word of the params among `args`, which are passed on only after it is set -- a
// dynamic-schedule slot when the CTAs loop over rows (work > grid), else null.
template <typename... KArgs, typename... Args>
inline int launch_persistent_pdl(void (*kern)(KArgs...), const char* what, int threads, size_t smem, long long work,
                                 int** sched, cudaStream_t st, const Args&... args) {
  int grid = 0;
  if (int rc = persistent_grid(kern, threads, smem, work, &grid)) return rc;
  if (sched) *sched = work > grid ? next_sched_slot() : nullptr;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3((unsigned)threads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
  return check_launch(what);
}

// Calls f(std::integral_constant<int, V>{}) for the run-time value v in [LO, HI] and returns its result; returns
// `otherwise` for any other v.  Fans a run-time size out to the kernel instantiation for it.
template <int LO, int HI, typename F>
inline int with_int(int v, F&& f, int otherwise = kUnsupported) {
  if constexpr (LO <= HI) {
    if (v == LO) return f(std::integral_constant<int, LO>{});
    return with_int<LO + 1, HI>(v, f, otherwise);
  } else {
    return otherwise;
  }
}

// The direct-DFT kernels (Clifford and bind) keep a row's transform in shared memory: longer rows are refused.
constexpr size_t kGenericSmemLimit = 200 * 1024;

inline bool is_pow2(long long x) { return x > 0 && (x & (x - 1)) == 0; }
inline int ilog2(long long x) { int l = 0; while ((1LL << l) < x) ++l; return l; }
inline bool aligned(const void* p, size_t a) { return (reinterpret_cast<uintptr_t>(p) % a) == 0; }

}  // namespace cvb
